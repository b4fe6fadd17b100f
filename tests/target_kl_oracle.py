"""SB3's ``target_kl`` early stopping (``PPO.train``), restated on top of the PPO oracles for ``PPOAgent(target_kl=...)``.

For every minibatch in order SB3 computes the loss and its gradient, appends the minibatch's loss terms, KL and clip
fraction to the update's records, and then, if ``approx_kl > 1.5 * target_kl`` (strictly), stops: that minibatch's
optimizer step is not taken and neither is any later one of the update.  ``update`` walks a given sequence of minibatches
(all epochs, flattened) that way with ``loss_fn(flat, i)`` giving the oracle dict of minibatch i (``oracle.ppo_ref.
loss_and_grad`` or ``oracle.ppo_categorical_ref.loss_and_grad`` on its rows, or a stand-in) and ``oracle.ppo_ref.
clip_adam`` for the step.  The oracles themselves are not modified.
"""
from oracle import ppo_ref


def stops(approx_kl, target_kl):
    """SB3's test: strictly above 1.5 target_kl (never with target_kl None)."""
    return target_kl is not None and approx_kl > 1.5 * target_kl


def update(flat, m, v, step, count, loss_fn, target_kl, lr=3e-4, max_norm=0.5):
    """``count`` minibatches from Adam state (flat, m, v, step).  Returns dict(flat, m, v, step, records, steps,
    stopped): ``records`` holds the oracle dict of every minibatch that entered the metrics (0..the stopping one)."""
    records, steps, stopped = [], 0, False
    for i in range(count):
        r = loss_fn(flat, i)
        records.append(r)
        if stops(r["approx_kl"], target_kl):
            stopped = True
            break
        step += 1
        steps += 1
        flat, m, v, _ = ppo_ref.clip_adam(flat, r["grad"], m, v, step, lr=lr, max_norm=max_norm)
    return dict(flat=flat, m=m, v=v, step=step, records=records, steps=steps, stopped=stopped)
