"""Host-buffer rollout loop: observations, actions, rewards and flags live in page-locked HOST memory.

This is the shape of the reference's loop (``training/routine.py:127-147``: the policy sees a host observation, the
env receives a host action and returns host results) for E lock-step envs: per group of envs and per policy step

    pinned observation --H2D--> policy (3 tcgen05 GEMMs + heads / sampling) --> fused env step kernel
    action --D2H--> pinned;  observation / reward / terminated / truncated written by the step kernel straight into the
    pinned buffers (zero-copy, hrp_env_step_host_async)

captured ONCE as a CUDA graph per group (the sampling noise's draw counter is device-resident,
``hrp_ppo_act_sample_ctr``), so a group-step costs the host one graph launch and one event wait.  With G > 1 groups on
G streams, one group's PCIe traffic and host turn-around hide under the other groups' kernels.
"""
from __future__ import annotations

from typing import Any, Dict, List

import numpy as np
import torch

from .. import _lib


class HostBufferPipeline:
    """``groups``: HighwayVecEnv handles (their env counts may differ).  After ``reset(seed)``, ``launch(g)`` enqueues
    one policy step of group g and ``wait(g)`` returns once its results are in ``buffers[g]`` (numpy views of the
    pinned tensors: ``obs`` [E_g, N, F_out] -- both the policy's input and the step's output --, ``action`` [E_g, 2],
    ``reward``, ``terminated``, ``truncated`` [E_g])."""

    def __init__(self, agent, groups: List[Any], use_graphs: bool = True, kernel_fetch: bool = True, chunks: int = 1):
        """``chunks`` > 1: the observation is fetched in row chunks, one after the other, and the policy of a chunk runs
        (on its own stream and workspace lane) while the next chunk is still crossing PCIe; the env step waits for all."""
        self.agent, self.envs, self.use_graphs = agent, list(groups), bool(use_graphs)
        self.kernel_fetch, self._lib = bool(kernel_fetch), _lib.load()
        self.chunks = max(1, int(chunks))
        dev = agent.device
        self.groups: List[Dict[str, Any]] = []
        self.buffers: List[Dict[str, np.ndarray]] = []
        A = agent.actor_critic.action_dim
        pin = lambda *shape, dtype=torch.float32: torch.zeros(shape, dtype=dtype).pin_memory()
        for gi, env in enumerate(self.envs):
            Eg, S = env.num_envs, env.N * env.F_out
            g = {"env": env, "stream": torch.cuda.Stream(device=dev), "side": torch.cuda.Stream(device=dev),
                 "done": torch.cuda.Event(), "obs_h": pin(Eg, env.N, env.F_out), "act_h": pin(Eg, A), "rew_h": pin(Eg),
                 "te_h": pin(Eg, dtype=torch.uint8), "tr_h": pin(Eg, dtype=torch.uint8),
                 "obs_d": torch.empty((Eg, S), device=dev),
                 "out": {"action": torch.empty((Eg, A), device=dev), "pre_tanh": torch.empty((Eg, A), device=dev),
                         "log_prob": torch.empty(Eg, device=dev), "value": torch.empty(Eg, device=dev)},
                 "draw": agent.actor_critic.new_draw_counter(), "draw0": agent.actor_critic._draw, "steps": 0,
                 "graph": None, "version": None, "lane": 1 + gi * self.chunks,
                 # chunked only when the chunks are whole and 16-byte aligned (hrp_fetch_host)
                 "C": self.chunks if Eg % self.chunks == 0 and (Eg // self.chunks * S * 4) % 16 == 0 else 1,
                 "draws": [agent.actor_critic.new_draw_counter() for _ in range(self.chunks)],
                 "cstreams": [torch.cuda.Stream(device=dev) for _ in range(self.chunks - 1)],
                 "row_base": int(getattr(env, "env_id_base", 0)), "pending": False, "index": gi}
            self.groups.append(g)
            self.buffers.append({"obs": g["obs_h"].numpy(), "action": g["act_h"].numpy(), "reward": g["rew_h"].numpy(),
                                 "terminated": g["te_h"].numpy(), "truncated": g["tr_h"].numpy()})
        self.launches = 0   # kernels of this library enqueued (per group-step and chunk: [fetch,] 3 GEMMs, heads; + env step)

    def reset(self, seed: int) -> None:
        for g, b in zip(self.groups, self.buffers):
            g["env"].reset_host(seed, b["obs"])

    def _enqueue(self, g: Dict[str, Any]) -> None:
        """The work of one group-step on the current stream (captured, or issued eagerly)."""
        env, ac = g["env"], self.agent.actor_critic
        Eg, S = env.num_envs, env.N * env.F_out
        cur = torch.cuda.current_stream(self.agent.device)
        C = g["C"]
        rows = Eg // C
        fetched = []
        for c in range(C):       # the chunks cross PCIe one after the other, on the group's stream
            lo, hi = c * rows, (c + 1) * rows
            if self.kernel_fetch:    # H2D observation by a kernel (hrp_fetch_host): the first GEMM follows it within ~1 us
                _lib.check(self._lib.hrp_fetch_host(g["obs_d"][lo:hi].data_ptr(), g["obs_h"][lo:hi].data_ptr(), rows * S * 4,
                                                    cur.cuda_stream), "hrp_fetch_host")
            else:                    # ... or by the copy engine
                g["obs_d"][lo:hi].copy_(g["obs_h"][lo:hi].view(rows, S), non_blocking=True)
            if C > 1:
                ev = torch.cuda.Event()
                ev.record(cur)
                fetched.append(ev)
        joins = []
        for c in range(C):       # the policy of chunk c: rows [lo, hi), its own workspace lane, draw counter and stream
            lo, hi = c * rows, (c + 1) * rows
            ac.row_base = g["row_base"] + lo
            out = g["out"] if C == 1 else {k: v[lo:hi] for k, v in g["out"].items()}
            if c == C - 1:           # the last chunk stays on the group's stream (its fetch is the last one there)
                self.agent.act(g["obs_d"][lo:hi], out=out, lane=g["lane"] + c, draw_counter=g["draws"][c])
            else:
                st = g["cstreams"][c]
                st.wait_event(fetched[c])
                with torch.cuda.stream(st):
                    self.agent.act(g["obs_d"][lo:hi], out=out, lane=g["lane"] + c, draw_counter=g["draws"][c])
                    ev = torch.cuda.Event()
                    ev.record(st)
                joins.append(ev)
        for ev in joins:
            cur.wait_event(ev)
        ac.row_base = g["row_base"]
        acted = torch.cuda.Event()
        acted.record(cur)
        g["side"].wait_event(acted)
        with torch.cuda.stream(g["side"]):                                         # D2H action, under the env kernel
            g["act_h"].copy_(g["out"]["action"], non_blocking=True)
            copied = torch.cuda.Event()
            copied.record(g["side"])
        b = self.buffers[g["index"]]
        env.step_host_async(g["out"]["action"], b["obs"], b["reward"], b["terminated"], b["truncated"])
        cur.wait_event(copied)

    def launch(self, gi: int) -> None:
        g = self.groups[gi]
        if g["pending"]:
            self.wait(gi)
        # torch.cuda.set_stream, not the `with torch.cuda.stream(...)` context: entering and leaving the context each
        # cost a cudaGetDeviceCount (~15 us) -- host time during which the GPU of a one-group pipeline has nothing to do
        home = torch.cuda.current_stream(self.agent.device)
        torch.cuda.set_stream(g["stream"])
        try:
            if not self.use_graphs:
                self._enqueue(g)
            elif g["graph"] is None or g["version"] != g["env"].param_version:
                # a captured env step keeps the seed / masks of its capture: capture again after they changed
                self._enqueue(g)          # eager first: warms every kernel variant and the workspace lane
                g["stream"].synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=g["stream"]):
                    self._enqueue(g)
                g["graph"], g["version"] = graph, g["env"].param_version
            else:
                g["graph"].replay()
            g["done"].record(g["stream"])
        finally:
            torch.cuda.set_stream(home)
        g["pending"] = True
        g["steps"] += 1
        # keep the policy's host-side draw counter ahead of the device-resident ones: a later eager act() must not
        # repeat (seed, row, draw) triples this pipeline has used
        ac = self.agent.actor_critic
        ac._draw = max(ac._draw, g["draw0"] + g["steps"])
        self.launches += g["C"] * (4 + int(self.kernel_fetch)) + 1

    def wait(self, gi: int) -> Dict[str, np.ndarray]:
        g = self.groups[gi]
        if g["pending"]:
            g["done"].synchronize()
            g["pending"] = False
        return self.buffers[gi]

    def close(self) -> None:
        for gi in range(len(self.groups)):
            self.wait(gi)
        for g in self.groups:
            g["graph"] = None
