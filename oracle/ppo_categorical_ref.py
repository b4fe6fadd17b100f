"""oracle/ppo_categorical_ref.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Plain PyTorch (CPU, autograd) restatement of the categorical policy that ``hrp_ppo_create_ex(...,
HRP_PPO_CATEGORICAL, ...)`` runs: the trunk, critic, clipped surrogate, value MSE, entropy bonus,
clip_grad_norm_ and Adam of ``oracle/ppo_ref.py``, with the tanh-Gaussian head replaced by
``torch.distributions.Categorical(logits=actor_mean(x))``.  The functions mirror ``ppo_ref``'s: ``forward``,
``evaluate``, ``loss_and_grad`` and ``clip_adam``; they compute in the dtype of their inputs (fp32 or fp64).

NOT PINNED by any reference fixture: the reference (``ppo/agent.py``) has no discrete agent, so there is no
output of it to compare with.  This is the standard PPO-with-Categorical formulation, checked against torch
itself (``tests/test_categorical_cpu.py``: fp32 against fp64, and a finite-difference gradient check).

Only ``tests/`` and ``tools/`` may import this module.
"""
import numpy as np
import torch
from torch.distributions import Categorical

from .ppo_ref import clip_adam  # noqa: F401  (the optimizer step does not depend on the head)


def shapes(S, n, H):
    """The flat layout: ppo_ref.shapes without log_std, n logits in actor_mean.2."""
    return [("shared.0.weight", (H, S)), ("shared.0.bias", (H,)),
            ("shared.2.weight", (H, H)), ("shared.2.bias", (H,)),
            ("actor_mean.0.weight", (H, H)), ("actor_mean.0.bias", (H,)),
            ("actor_mean.2.weight", (n, H)), ("actor_mean.2.bias", (n,)),
            ("critic.0.weight", (H, H)), ("critic.0.bias", (H,)),
            ("critic.2.weight", (1, H)), ("critic.2.bias", (1,))]


def param_count(S, n, H):
    return sum(int(np.prod(s)) for _, s in shapes(S, n, H))


def unflatten(flat, S, n, H):
    out, off = {}, 0
    for name, shp in shapes(S, n, H):
        k = int(np.prod(shp))
        out[name] = flat[off:off + k].view(shp)
        off += k
    assert off == flat.numel()
    return out


def forward(flat, x, S, n, H):
    """(logits [B, n], value [B, 1])"""
    p = unflatten(flat, S, n, H)
    h = torch.relu(x @ p["shared.0.weight"].T + p["shared.0.bias"])
    h = torch.relu(h @ p["shared.2.weight"].T + p["shared.2.bias"])
    a = torch.relu(h @ p["actor_mean.0.weight"].T + p["actor_mean.0.bias"])
    logits = a @ p["actor_mean.2.weight"].T + p["actor_mean.2.bias"]
    c = torch.relu(h @ p["critic.0.weight"].T + p["critic.0.bias"])
    value = c @ p["critic.2.weight"].T + p["critic.2.bias"]
    return logits, value


def evaluate(flat, x, ids, S, n, H):
    """log_softmax(logits)[id], value, the state-dependent entropy -sum p log p"""
    logits, value = forward(flat, x, S, n, H)
    dist = Categorical(logits=logits)
    ids = torch.as_tensor(ids).reshape(-1).long()
    return dist.log_prob(ids), value, dist.entropy()


def loss_and_grad(flat, x, ids, old_logp, adv, ret, S, n, H, eps_clip=0.2, value_coef=0.5, entropy_coef=0.005):
    """The clipped surrogate + value MSE - entropy bonus of ppo_ref.loss_and_grad; same return dict."""
    flat = flat.detach().clone().requires_grad_(True)
    logp, value, ent = evaluate(flat, x, ids, S, n, H)
    ratio = torch.exp(logp - old_logp)
    s1, s2 = ratio * adv, torch.clamp(ratio, 1 - eps_clip, 1 + eps_clip) * adv
    actor = -torch.min(s1, s2).mean()
    critic = torch.nn.functional.mse_loss(value.squeeze(-1), ret)
    loss = actor + value_coef * critic - entropy_coef * ent.mean()
    loss.backward()
    with torch.no_grad():
        lr_ = logp - old_logp
        kl = ((torch.exp(lr_) - 1) - lr_).mean()
        cf = (torch.abs(ratio - 1) > eps_clip).to(flat.dtype).mean()
    return dict(loss=float(loss.detach()), actor=float(actor.detach()), critic=float(critic.detach()),
                entropy=float(ent.mean().detach()),
                clip_fraction=float(cf), approx_kl=float(kl), grad=flat.grad.detach().clone())


def sample(probs, u):
    """Inverse-CDF draw of the kernels: the first j with u < sum_{i<=j} p_i, n - 1 if there is none.  probs [B, n],
    u [B] (numpy).  Returns (ids, distance of u to the nearest cumulative boundary)."""
    cdf = np.cumsum(probs, axis=1)
    ids = np.minimum((u[:, None] >= cdf).sum(1), probs.shape[1] - 1)
    return ids, np.abs(cdf[:, :-1] - u[:, None]).min(1) if probs.shape[1] > 1 else np.full(len(u), np.inf)
