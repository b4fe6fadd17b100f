"""Peer-memory fused reduce + clip + Adam (hrp_clip_adam_step_p2p) against the NCCL all-reduce + hrp_clip_adam_step
pair, on the same per-rank minibatches.  Run with one rank per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/p2p_check.py

World size 2: the two-term sums are commutative, so the parameters must agree BIT FOR BIT after every step.  More
ranks: NCCL's reduction order differs from rank order, so the summed GRADIENT of the first step is compared (1e-5 of
its max-abs; Adam turns last-bit differences of near-zero gradients into +-lr parameter moves, which makes the
parameters themselves a poor yardstick).  Every rank must hold identical parameters at the end in any case.

``--bootstrap-truncated``: the graph-replayed updates run on rollouts collected with time-limit bootstrapping
(final_value of truncated steps, hrp_gae_ex); GAE is per env, so the sharded update needs no other exchange.

``--ppo-options``: three more graph-replayed updates each with the peer-memory exchange and with the NCCL all-reduce,
with the clipped value loss (clip_value) and a linearly annealed learning rate in device memory (set_lr before every
update): the ranks must agree bit for bit, and the minibatch graphs must be captured once."""
import os
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from highway_rope_ppo_b200.ppo.agent import PPOAgent  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
S, A, H, B, steps = 60, 2, 256, 4096, 24
BOOT = "--bootstrap-truncated" in sys.argv
OPTS = "--ppo-options" in sys.argv


def make(p2p: bool) -> PPOAgent:
    torch.manual_seed(0)
    a = PPOAgent(S, A, lr=3e-4, hidden_dim=H, batch_size=B, epochs=1, device=dev)
    a.use_p2p = p2p
    return a


p2p, ref = make(True), make(False)
assert p2p._ensure_comm(world), "peer-memory exchange could not be set up"
g = torch.Generator(device=dev).manual_seed(100 + rank)   # every rank its own shard of the minibatch
t_p2p = t_ref = 0.0
grad_err = 0.0
for it in range(steps):
    flat = {"states": torch.randn(B, S, generator=g, device=dev) * 0.5, "pre_tanh": torch.randn(B, A, generator=g, device=dev),
            "log_prob": torch.randn(B, generator=g, device=dev) * 0.1 - 2.0, "adv": torch.randn(B, generator=g, device=dev),
            "ret": torch.randn(B, generator=g, device=dev)}
    for agent in (p2p, ref):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        agent._minibatch_step(flat, None, B, world)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if it >= 4:
            if agent is p2p:
                t_p2p += dt
            else:
                t_ref += dt
    if it == 0:
        # summed gradient of the first step (parity 0): the exported allocation is [grad 0 | grad 1 | sum 0 | sum 1 | flags]
        P = p2p.actor_critic.num_params
        pad = (P + 31) // 32 * 32

        class _Raw:
            __cuda_array_interface__ = {"shape": (P,), "typestr": "<f4", "data": (p2p._grad_parity[0].data_ptr() + 4 * 2 * pad, False),
                                        "version": 2}

        keep = _Raw()
        gsum = torch.as_tensor(keep, device=dev)
        grad_err = ((gsum - ref.grad).abs().max() / ref.grad.abs().max()).item()
a, b = p2p.actor_critic.flat, ref.actor_critic.flat
diff = (a - b).abs().max().item()
same = torch.equal(a, b)
gathered = [torch.empty_like(a) for _ in range(world)]
dist.all_gather(gathered, a)
ranks_equal = all(torch.equal(gathered[0], x) for x in gathered)
moved = (a - make(False).actor_critic.flat).abs().max().item()
if rank == 0:
    print(f"world {world}: {steps} optimizer steps; |p2p - nccl| max {diff:.3e} (bit-identical: {same}); identical on every rank: "
          f"{ranks_equal}; summed gradient of step 0 differs by {grad_err:.2e} of its max; parameters moved by {moved:.3e}; eager step {t_p2p / (steps - 4) * 1e6:.0f} us (p2p) vs "
          f"{t_ref / (steps - 4) * 1e6:.0f} us (nccl)")
ok = ranks_equal and moved > 1e-4 and grad_err < 1e-5 and (same if world == 2 else True)

# ---- PPOAgent.update through CUDA graphs: 3 minibatches x 3 epochs (an odd number of steps per epoch, so the same
# minibatch is replayed with both parities of the double-buffered exchange), two updates
def rollout(agent, seed):
    T, E = 6, 2048
    gg = torch.Generator(device=dev).manual_seed(seed)
    r = agent.memory.begin_rollout(T, E, S, A, bootstrap_truncated=BOOT)
    r["states"].copy_(torch.randn(T + 1, E, S, generator=gg, device=dev) * 0.5)
    r["pre_tanh"].copy_(torch.randn(T, E, A, generator=gg, device=dev))
    r["action"].copy_(torch.tanh(r["pre_tanh"]))
    r["log_prob"].copy_(torch.randn(T, E, generator=gg, device=dev) * 0.1 - 2.0)
    r["value"].copy_(torch.randn(T, E, generator=gg, device=dev))
    r["reward"].copy_(torch.rand(T, E, generator=gg, device=dev))
    r["done"].copy_((torch.rand(T, E, generator=gg, device=dev) < 0.05).to(torch.uint8))
    if BOOT:
        r["terminated"].copy_(r["done"])
        r["truncated"].copy_((torch.rand(T, E, generator=gg, device=dev) < 0.1).to(torch.uint8))
        r["final_value"].copy_(torch.randn(T, E, generator=gg, device=dev))
        r["done"].copy_(r["terminated"] | r["truncated"])


torch.manual_seed(1)
upd = PPOAgent(S, A, lr=3e-4, hidden_dim=H, batch_size=B, epochs=3, device=dev)
import numpy as np  # noqa: E402

for u in range(2):
    rollout(upd, 1000 + 10 * u + rank)
    np.random.seed(5 + u)          # the same minibatch permutation on every rank
    upd.update(last_value=0.0)
flat = upd.actor_critic.flat
gathered = [torch.empty_like(flat) for _ in range(world)]
dist.all_gather(gathered, flat)
upd_equal = all(torch.equal(gathered[0], x) for x in gathered)
if rank == 0:
    print(f"world {world}: two graph-replayed updates (18 optimizer steps, both parities"
          f"{', bootstrapped truncation' if BOOT else ''}): identical on every rank: {upd_equal}; "
          f"exchange: {'peer-memory kernel' if upd._comm is not None else 'nccl'}; graphs captured: {len(upd._graph_state['graphs'])}")
ok = ok and upd_equal
upd.close()
if OPTS:
    from highway_rope_ppo_b200.training.routine import linear_lr

    for use_p2p in (True, False):
        torch.manual_seed(2)
        agent = PPOAgent(S, A, lr=3e-4, hidden_dim=H, batch_size=B, epochs=3, device=dev, clip_value=0.2)
        agent.use_p2p = use_p2p
        states = []
        for u in range(3):
            rollout(agent, 2000 + 10 * u + rank)
            agent.set_lr(linear_lr(3e-4, u, 3))
            np.random.seed(7 + u)
            agent.update(last_value=0.0)
            st = agent._graph_state
            states.append((id(st), sorted(id(x) for x in st["graphs"].values())))
        flat = agent.actor_critic.flat
        gathered = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        eq = all(torch.equal(gathered[0], x) for x in gathered)
        once = states[0] == states[1] == states[2]
        if rank == 0:
            print(f"world {world}: anneal_lr + clip_value, three graph-replayed updates, exchange "
                  f"{'peer-memory kernel' if agent._comm is not None else 'nccl'}: identical on every rank: {eq}; "
                  f"graphs captured once: {once}")
        ok = ok and eq and once
        agent.close()
p2p.close()
dist.barrier()
sys.stdout.flush()
# communicator teardown (it was seen to hang after NCCL work captured in graphs; with the peer-memory exchange no NCCL
# work is captured): give it 20 s
import threading  # noqa: E402

threading.Timer(20.0, lambda: (print("destroy_process_group did not return within 20 s", flush=True), os._exit(0 if ok else 1))).start()
dist.destroy_process_group()
if rank == 0:
    print("destroy_process_group returned", flush=True)
os._exit(0 if ok else 1)
