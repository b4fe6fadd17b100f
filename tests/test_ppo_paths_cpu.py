"""The TF32 twin of the PPO oracles (tests/tf32_twin.py), which sets the math-mode-1 tolerances of
tests/test_ppo_paths_gpu.py: with the truncation off it is the oracle bit for bit; with it on it truncates exactly the
operands of the four hidden Linear layers, forward and backward, and nothing else; its ``trunc`` is the one
tools/tf32_probe.py measured the tensor cores against."""
import ast
import contextlib
import os

import numpy as np
import pytest
import torch

import tf32_twin
from oracle import ppo_categorical_ref as cref
from oracle import ppo_ref
from ppo_options_oracle import loss_and_grad, loss_and_grad_cat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _probe_trunc():
    """``trunc`` as tools/tf32_probe.py defines it (the script itself needs a GPU, so only the function is taken)."""
    path = os.path.join(ROOT, "tools", "tf32_probe.py")
    tree = ast.parse(open(path).read())
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "trunc")
    ns = {"torch": torch}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
    return ns["trunc"]


# (value, its TF32 truncation): 10 mantissa bits kept, the rest dropped toward zero, either sign
HAND = [(1.0, 1.0), (1.0 + 2 ** -10, 1.0 + 2 ** -10), (1.0 + 2 ** -11, 1.0), (1.0 + 2 ** -10 + 2 ** -11, 1.0 + 2 ** -10),
        (2.0 - 2 ** -23, 2.0 - 2 ** -10), (-(1.0 + 2 ** -11 + 2 ** -12), -1.0), (3.0 * 2 ** -100, 3.0 * 2 ** -100),
        (0.0, 0.0), (2 ** -149, 0.0), (3.0 + 2 ** -22, 3.0), (-(2.0 ** 100) * (1 + 2 ** -9 + 2 ** -20), -(2.0 ** 100) * (1 + 2 ** -9)),
        (0.1, 0.0999755859375), (-0.1, -0.0999755859375), (float("inf"), float("inf"))]


def test_trunc_matches_the_probe_on_hand_picked_values():
    probe = _probe_trunc()
    x = torch.tensor([v for v, _ in HAND], dtype=torch.float32)
    want = torch.tensor([t for _, t in HAND], dtype=torch.float32)
    assert torch.equal(tf32_twin.trunc(x), want)
    assert torch.equal(probe(x), want)
    r = torch.randn(10000, generator=torch.Generator().manual_seed(0)) * 1e3
    assert torch.equal(tf32_twin.trunc(r), probe(r))
    # fp64 operands: rounded to fp32 first, as the kernel's buffers hold them
    d = torch.tensor([1.0 + 2 ** -11 + 2 ** -30, 1.0 + 2 ** -10 - 2 ** -40], dtype=torch.float64)
    assert tf32_twin.trunc64(d).tolist() == [1.0, 1.0 + 2 ** -10]


def _flat(S, A, H, discrete, seed):
    g = torch.Generator().manual_seed(seed)
    n = sum(int(np.prod(s)) for _, s in (cref if discrete else ppo_ref).shapes(S, A, H))
    return (torch.rand(n, generator=g, dtype=torch.float64) * 2 - 1) / np.sqrt(min(S, H))


def _batch(S, A, B, discrete, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, S, generator=g, dtype=torch.float64) * 0.5
    act = torch.randint(0, A, (B,), generator=g) if discrete else torch.randn(B, A, generator=g, dtype=torch.float64)
    old, adv, R, vo = (torch.randn(B, generator=g, dtype=torch.float64) for _ in range(4))
    return x, act, old, adv, R, vo


@pytest.mark.parametrize("discrete,A", [(False, 1), (False, 3), (True, 2), (True, 8)])
@pytest.mark.parametrize("S,H,B", [(7, 16, 5), (60, 96, 33), (25, 102, 40)])
def test_twin_without_truncation_is_the_oracle_bit_for_bit(discrete, A, S, H, B):
    flat = _flat(S, A, H, discrete, S + H)
    x, act, old, adv, R, vo = _batch(S, A, B, discrete, B)
    ref = cref if discrete else ppo_ref
    fn = loss_and_grad_cat if discrete else loss_and_grad
    outs = []
    for twin in (False, True):
        ctx = tf32_twin.tf32(H, truncate=False) if twin else contextlib.nullcontext()
        with ctx:
            fwd = ref.forward(flat, x, S, A, H)
            ev = ref.evaluate(flat, x, act, S, A, H)
            plain = fn(flat, x, act, old, adv, R, S, A, H)
            clipped = fn(flat, x, act, old, adv, R, S, A, H, old_value=vo, clip_value=0.3)
        outs.append((fwd, ev, plain, clipped))
    (f0, e0, p0, c0), (f1, e1, p1, c1) = outs
    for a, b in zip(list(f0) + list(e0), list(f1) + list(e1)):
        assert torch.equal(a, b)
    for r0, r1 in ((p0, p1), (c0, c1)):
        assert r0.keys() == r1.keys()
        for k in r0:
            assert torch.equal(r0[k], r1[k]) if k == "grad" else r0[k] == r1[k], k


def _manual_forward(flat, x, S, A, H):
    """ppo_ref.forward with trunc64 on both operands of the four hidden layers, written out."""
    p = ppo_ref.unflatten(flat, S, A, H)
    q = tf32_twin.trunc64
    lin = lambda h, w, b: q(h) @ q(p[w]).T + p[b]
    h = torch.relu(lin(x, "shared.0.weight", "shared.0.bias"))
    h = torch.relu(lin(h, "shared.2.weight", "shared.2.bias"))
    a = torch.relu(lin(h, "actor_mean.0.weight", "actor_mean.0.bias"))
    c = torch.relu(lin(h, "critic.0.weight", "critic.0.bias"))
    return a @ p["actor_mean.2.weight"].T + p["actor_mean.2.bias"], c @ p["critic.2.weight"].T + p["critic.2.bias"]


def test_twin_truncates_the_hidden_layers_and_not_the_heads():
    S, A, H, B = 13, 3, 24, 37
    flat = _flat(S, A, H, False, 1)
    x = _batch(S, A, B, False, 2)[0]
    with tf32_twin.tf32(H):
        mean, _, value = ppo_ref.forward(flat, x, S, A, H)
    m2, v2 = _manual_forward(flat, x, S, A, H)
    assert torch.equal(mean, m2) and torch.equal(value, v2)
    m0, _, v0 = ppo_ref.forward(flat, x, S, A, H)
    d = float((mean - m0).abs().max())
    assert 1e-6 < d < 1e-2   # of the size TF32 operands give, not zero


def test_twin_backward_truncates_both_gemm_operands():
    """d/dx and d/dW of x @ W^T inside the twin are trunc(g) trunc(W) and trunc(g)^T trunc(x)."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(9, 11, generator=g, dtype=torch.float64).requires_grad_(True)
    W = torch.randn(20, 11, generator=g, dtype=torch.float64).requires_grad_(True)
    gy = torch.randn(9, 20, generator=g, dtype=torch.float64)
    with tf32_twin.tf32(20):
        y = x @ W.T
    y.backward(gy)
    q = tf32_twin.trunc64
    assert torch.equal(y.detach(), q(x.detach()) @ q(W.detach()).T)
    assert torch.allclose(x.grad, q(gy) @ q(W.detach()), rtol=1e-14, atol=0)
    assert torch.allclose(W.grad, q(gy).T @ q(x.detach()), rtol=1e-14, atol=0)
    assert not torch.allclose(x.grad, gy @ W.detach(), rtol=1e-6, atol=0)
    # a product with another width (a head) passes through untouched
    with tf32_twin.tf32(21):
        y2 = (x @ W.T).detach()
    assert torch.equal(y2, x.detach() @ W.detach().T)
