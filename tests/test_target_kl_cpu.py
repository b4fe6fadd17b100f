"""CPU checks of target_kl early stopping: SB3's loop as the oracle restates it, on hand-worked KL sequences and on a
real tiny network, and the argument errors of ``PPOAgent(target_kl=...)`` and of the new C entry points that are
reachable without a device."""
import ctypes as C
import math

import pytest
import torch

from oracle import ppo_ref
from target_kl_oracle import stops, update


def _fake(kls, P=3):
    """A loss_fn whose minibatch i has approx_kl kls[i] and gradient (i + 1) * ones."""
    def fn(flat, i):
        return {"approx_kl": kls[i], "loss": float(i), "grad": torch.full((P,), float(i + 1), dtype=torch.float64)}
    return fn


def _run(kls, target_kl):
    P = 3
    z = torch.zeros(P, dtype=torch.float64)
    return update(torch.ones(P, dtype=torch.float64), z, z.clone(), 0, len(kls), _fake(kls, P), target_kl)


def test_stop_at_the_first_minibatch_takes_no_step():
    r = _run([0.031, 0.0, 0.0], 0.02)   # limit 0.03
    assert r["stopped"] and r["steps"] == 0 and r["step"] == 0 and len(r["records"]) == 1
    assert torch.equal(r["flat"], torch.ones(3, dtype=torch.float64)) and not r["m"].any()


def test_stop_mid_epoch_keeps_the_stopping_minibatch_in_the_records():
    r = _run([0.001, 0.01, 0.029, 0.04, 0.001, 0.0], 0.02)
    assert r["stopped"] and r["steps"] == 3 and r["step"] == 3
    assert [q["loss"] for q in r["records"]] == [0.0, 1.0, 2.0, 3.0]
    # the same as three plain Adam steps
    P = 3
    flat, m, v = torch.ones(P, dtype=torch.float64), torch.zeros(P, dtype=torch.float64), torch.zeros(P, dtype=torch.float64)
    for i in range(3):
        flat, m, v, _ = ppo_ref.clip_adam(flat, torch.full((P,), float(i + 1), dtype=torch.float64), m, v, i + 1)
    assert torch.equal(r["flat"], flat) and torch.equal(r["m"], m) and torch.equal(r["v"], v)


def test_kl_exactly_at_the_limit_does_not_stop():
    t = 0.02
    limit = 1.5 * t
    assert not stops(limit, t) and stops(math.nextafter(limit, 1.0), t)
    r = _run([limit, limit, limit], t)
    assert not r["stopped"] and r["steps"] == 3 and len(r["records"]) == 3


def test_no_stop_and_no_target_kl():
    for t in (None, 1.0):
        r = _run([0.5, 0.9, 1.4], t)
        assert not r["stopped"] and r["steps"] == 3 and r["step"] == 3


def test_real_network_kl_grows_until_the_stop():
    """The oracle on a tiny Gaussian network: one minibatch stepped repeatedly moves the policy away from the rollout's,
    so its KL grows from 0; a limit between two recorded values stops exactly at the first one above it."""
    S, A, H, B = 3, 2, 4, 16
    g = torch.Generator().manual_seed(0)
    n = sum(math.prod(s) for _, s in ppo_ref.shapes(S, A, H))
    flat = torch.randn(n, generator=g, dtype=torch.float64) * 0.3
    x = torch.randn(B, S, generator=g, dtype=torch.float64)
    mean, _, _ = ppo_ref.forward(flat, x, S, A, H)
    z = mean.detach() + torch.randn(B, A, generator=g, dtype=torch.float64)
    old = ppo_ref.evaluate(flat, x, z, S, A, H)[0].detach()
    adv = torch.randn(B, generator=g, dtype=torch.float64)
    ret = torch.randn(B, generator=g, dtype=torch.float64)
    fn = lambda f, i: ppo_ref.loss_and_grad(f, x, z, old, adv, ret, S, A, H)
    z0 = torch.zeros(n, dtype=torch.float64)
    free = update(flat, z0, z0.clone(), 0, 8, lambda f, i: dict(fn(f, i)), None, lr=3e-2)
    kls = [q["approx_kl"] for q in free["records"]]
    assert kls[0] < 1e-12 and kls[-1] > kls[1] > 0
    k = max(range(1, 8), key=lambda j: kls[j] - max(kls[:j]))
    assert kls[k] > max(kls[:k])
    t = (max(kls[:k]) + kls[k]) / 2 / 1.5
    r = update(flat, z0, z0.clone(), 0, 8, fn, t, lr=3e-2)
    assert r["stopped"] and r["steps"] == k and len(r["records"]) == k + 1
    assert torch.equal(r["flat"], update(flat, z0, z0.clone(), 0, k, fn, None, lr=3e-2)["flat"])


@pytest.mark.parametrize("bad", [0, 0.0, -0.01, float("nan"), float("inf"), "x", True, [0.1]])
def test_target_kl_value_errors_before_any_device_work(bad):
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    with pytest.raises(ValueError, match="target_kl"):
        PPOAgent(4, 2, target_kl=bad, device="cpu")


def _lib():
    from highway_rope_ppo_b200 import _lib

    return _lib.load(), _lib.last_error


def test_loss_grad_kl_argument_errors():
    lib, err = _lib()
    one = C.c_void_p(16)
    base = [one] * 8 + [64, 0.2, 0.5, 0.005, 1.0 / 64]
    assert lib.hrp_ppo_loss_grad_kl(*base, None, 0.0, one, None, one, one, None) == -1
    assert "stop_dev" in err()
    assert lib.hrp_ppo_loss_grad_kl(*base, None, 0.0, None, one, one, one, None) == -1
    assert "kl_out_dev" in err()
    assert lib.hrp_ppo_loss_grad_kl(*base, one, float("nan"), one, one, one, one, None) == -1
    assert "value_clip" in err()
    assert lib.hrp_ppo_loss_grad_kl(None, *base[1:], None, 0.0, one, one, one, one, None) == -1
    assert "null argument" in err()


def test_clip_adam_step_kl_argument_errors():
    lib, err = _lib()
    one = C.c_void_p(16)
    head = [one] * 5 + [100, 3e-4, None, 0.9, 0.999, 1e-8, 0.5, one]
    for kl, stop, limit, field in ((one, None, 0.03, "stop_dev"), (None, one, 0.03, "kl_dev"), (one, one, 0.0, "kl_limit"),
                                   (one, one, float("inf"), "kl_limit"), (one, one, -1.0, "kl_limit")):
        assert lib.hrp_clip_adam_step_kl(*head, kl, stop, limit, None) == -1
        assert field in err()
    assert lib.hrp_clip_adam_step_kl(*head[:5], 0, *head[6:], one, one, 0.03, None) == -1 and "bad argument n" in err()
    assert lib.hrp_clip_adam_step_p2p_kl(None, one, one, one, one, 3e-4, None, 0.9, 0.999, 1e-8, 0.5, one, one, 0.03,
                                         None) == -1
    assert "comm" in err()


def test_graph_if_argument_errors():
    lib, err = _lib()
    one = C.c_void_p(16)
    out = C.c_void_p()
    for args, field in (((None, one, one, C.byref(out)), "body_graph"), ((one, None, one, C.byref(out)), "stop_dev"),
                        ((one, one, None, C.byref(out)), "opened_dev"), ((one, one, one, None), "out")):
        assert lib.hrp_graph_if_create(*args) == -1
        assert field in err()
    assert lib.hrp_graph_if_launch(None, None) == -1 and "wrapped" in err()
    assert lib.hrp_graph_if_destroy(None) == 0
