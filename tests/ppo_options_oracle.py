"""The clipped value loss of ``PPOAgent(clip_value=...)`` / ``hrp_ppo_loss_grad_ex``, restated on top of the PPO oracles.

``loss_and_grad`` and ``loss_and_grad_cat`` are ``oracle.ppo_ref.loss_and_grad`` and ``oracle.ppo_categorical_ref.
loss_and_grad`` with two more arguments, ``old_value`` (the rollout's value of each sample) and ``clip_value`` (c).  With
both given, the value term of every sample is

    max((v - R)^2, (v_old + clamp(v - v_old, -c, c) - R)^2)

weighted like the reference's value MSE (``value_coef`` * the minibatch mean, no 1/2), and the gradient is torch
autograd's on that expression, in the dtype of the inputs.  Without them they ARE the oracles' functions, so every
existing comparison is unchanged.  The oracles themselves are not modified: ``oracle/`` restates the reference, which
has no clipped value loss.
"""
import torch

from oracle import ppo_categorical_ref as cref
from oracle import ppo_ref


def value_term(v, old_value, ret, clip_value):
    """Per-sample clipped value term (torch ops, autograd-able)."""
    v_clip = old_value + torch.clamp(v - old_value, -clip_value, clip_value)
    return torch.maximum((v - ret) ** 2, (v_clip - ret) ** 2)


def _loss_and_grad(evaluate, flat, x, act, old_logp, adv, ret, S, A, H, eps_clip, value_coef, entropy_coef, old_value,
                   clip_value):
    flat = flat.detach().clone().requires_grad_(True)
    logp, value, ent = evaluate(flat, x, act, S, A, H)
    ratio = torch.exp(logp - old_logp)
    s1, s2 = ratio * adv, torch.clamp(ratio, 1 - eps_clip, 1 + eps_clip) * adv
    actor = -torch.min(s1, s2).mean()
    critic = value_term(value.squeeze(-1), old_value, ret, clip_value).mean()
    loss = actor + value_coef * critic - entropy_coef * ent.mean()
    loss.backward()
    with torch.no_grad():
        lr_ = logp - old_logp
        kl = ((torch.exp(lr_) - 1) - lr_).mean()
        cf = (torch.abs(ratio - 1) > eps_clip).to(flat.dtype).mean()
    return dict(loss=float(loss.detach()), actor=float(actor.detach()), critic=float(critic.detach()),
                entropy=float(ent.mean().detach()),
                clip_fraction=float(cf), approx_kl=float(kl), grad=flat.grad.detach().clone())


def loss_and_grad(flat, x, z, old_logp, adv, ret, S, A, H, eps_clip=0.2, value_coef=0.5, entropy_coef=0.005,
                  old_value=None, clip_value=None):
    """The Gaussian policy (``oracle.ppo_ref``); same return dict."""
    if old_value is None and clip_value is None:
        return ppo_ref.loss_and_grad(flat, x, z, old_logp, adv, ret, S, A, H, eps_clip, value_coef, entropy_coef)
    return _loss_and_grad(ppo_ref.evaluate, flat, x, z, old_logp, adv, ret, S, A, H, eps_clip, value_coef, entropy_coef,
                          old_value, clip_value)


def loss_and_grad_cat(flat, x, ids, old_logp, adv, ret, S, n, H, eps_clip=0.2, value_coef=0.5, entropy_coef=0.005,
                      old_value=None, clip_value=None):
    """The categorical policy (``oracle.ppo_categorical_ref``); same return dict."""
    if old_value is None and clip_value is None:
        return cref.loss_and_grad(flat, x, ids, old_logp, adv, ret, S, n, H, eps_clip, value_coef, entropy_coef)
    return _loss_and_grad(cref.evaluate, flat, x, ids, old_logp, adv, ret, S, n, H, eps_clip, value_coef, entropy_coef,
                          old_value, clip_value)
