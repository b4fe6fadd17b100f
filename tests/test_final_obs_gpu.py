"""GPU checks of the final-observation output of the step kernel (hrp_env_step_final), the bootstrapped GAE
(hrp_gae_ex) and the batched loop that uses them (collect_rollout / update with bootstrap_truncated=True).

* The final observation of every finished env equals, bit for bit, the observation an autoreset = 0 twin returns from
  the same state and actions -- fp32 and fp64 kernels, sorted / shuffled / injected row order, RoPE / DistPE / RankPE,
  continuous and meta-action ego, crashes and time limits (on the same step too), with and without a step mask.
* Turning the output on changes nothing else: observation, reward, flags and the whole state after the step
  (episode and shuffle counters included) equal a plain step bit for bit; rows of unfinished and masked envs keep a
  NaN sentinel.
* hrp_gae_ex equals the fp64 oracle (oracle/gae_bootstrap.py) with NaN planted in every final_value row it must not
  read, and is bit-identical to hrp_gae when nothing is truncated.
* The rollout: graph replay equals the eager rollout, the flag leaves states / actions / rewards / flags unchanged,
  final_value is the critic of final_states, update's advantages are the oracle's, and a plain rollout after a
  bootstrapped one is back to the reference's semantics.
"""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import gae_bootstrap as gb
from oracle import ppo_ref

pytestmark = pytest.mark.gpu

_STATE = ("x", "y", "heading", "speed", "target_speed", "delta", "timer", "impact_x", "impact_y", "lane",
          "target_lane", "crashed", "has_impact", "time", "episode", "obs_draw")


def _cfg(highway_config, order, meta, duration=5):
    cfg = copy.deepcopy(highway_config)
    cfg["observation"]["order"] = order
    cfg["duration"] = duration
    if meta:
        cfg["action"] = {"type": "DiscreteMetaAction"}
    return cfg


def _spec(cfg, embed):
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import embed_spec_for

    torch.manual_seed(11)
    cond = {"none": Condition.SORTED, "rope": Condition.SHUFFLED_ROPE, "dist": Condition.SHUFFLED_DISTPE,
            "rank": Condition.SHUFFLED_RANKPE}[embed]
    return embed_spec_for(cond, cfg, None if embed in ("none", "rope") else 4)


def _vec(cfg, E, spec, autoreset, real64):
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv

    return HighwayVecEnv(cfg, E, device="cuda:0", embed=spec, autoreset=autoreset, seed=5, real64=real64)


def _actions(rng, E, meta):
    if meta:
        a = np.zeros((E, 2), dtype=np.float32)
        a[:, 0] = rng.integers(0, 5, E)
        return a
    a = rng.uniform(-1, 1, (E, 2)).astype(np.float32)
    a[: E // 4, 1] = rng.choice([-1.0, 1.0], E // 4)   # hard steering: crashes and off-road episodes
    return a


CASES = [
    # (real64, order, embed, meta, masked)
    (False, "sorted", "none", False, False),
    (False, "shuffled", "rope", False, False),
    (False, "perm", "dist", False, True),
    (False, "shuffled", "rank", True, False),
    (False, "sorted", "rope", True, True),
    (True, "shuffled", "dist", False, False),
    (True, "perm", "rank", True, False),
    (True, "sorted", "rope", False, True),
]


@pytest.mark.parametrize("real64,order,embed,meta,masked", CASES,
                         ids=[f"{'f64' if c[0] else 'f32'}-{c[1]}-{c[2]}-{'meta' if c[3] else 'cont'}"
                              f"{'-mask' if c[4] else ''}" for c in CASES])
def test_final_obs_equals_autoreset0_twin_and_changes_nothing_else(highway_config, real64, order, embed, meta,
                                                                    masked):
    """Three handles from one state every step: A steps with the final-observation output, B is A without it, Z is an
    autoreset = 0 twin.  final_obs[e] of every finished env == Z's obs[e]; A and B agree on everything else."""
    E, steps = (96 if real64 else 256), 6
    cfg = _cfg(highway_config, "shuffled" if order == "perm" else order, meta)
    spec = _spec(cfg, embed)
    A, B, Z = (_vec(cfg, E, spec, ar, real64) for ar in (True, True, False))
    for h in (A, B, Z):
        h.reset(5)   # the handle seed keys respawns and shuffle draws
    rng = np.random.default_rng(1)
    st = A.get_state()
    st["time"][:] = rng.integers(0, 5, E).astype(np.float64)   # time limits spread over the steps
    st["crashed"][:8, 0] = 1        # egos that crash on the first step: 0-3 on their last step (both flags), 4-7 not
    st["time"][:4], st["time"][4:8] = 4.0, 0.0
    A.set_state(st)
    N, F = A.N, A.F_out
    mask = torch.ones(E, dtype=torch.uint8, device="cuda:0")
    if masked:
        for h in (A, B, Z):
            h.set_step_mask(mask)
    counts = dict(term=0, trunc=0, both=0)
    for t in range(steps):
        st = A.get_state()
        B.set_state(st)
        Z.set_state(st)
        if masked:
            m = rng.random(E) < 0.7
            m[:8] |= t == 0
            mask.copy_(torch.from_numpy(m.astype(np.uint8)))
        a = torch.from_numpy(_actions(rng, E, meta)).cuda()
        perm = None
        if order == "perm":
            perm = torch.from_numpy(np.stack([rng.permutation(N - 1) for _ in range(E)]).astype(np.int32)).cuda()
        fin = torch.full((E, N, F), float("nan"), device="cuda:0")
        rows_a = torch.full((E, N), -7, dtype=torch.int32, device="cuda:0")
        rows_b = torch.full((E, N), -7, dtype=torch.int32, device="cuda:0")
        oa, ra, ta, ua = (x.clone() for x in A.step(a, perm=perm, row_vehicle=rows_a, final_obs_out=fin))
        ob, rb, tb, ub = (x.clone() for x in B.step(a, perm=perm, row_vehicle=rows_b))
        oz, rz, tz, uz = (x.clone() for x in Z.step(a, perm=perm))
        torch.cuda.synchronize()
        # nothing else changes
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(ta, tb) and torch.equal(ua, ub), t
        assert torch.equal(rows_a, rows_b), t
        sa, sb = A.get_state(), B.get_state()
        for k in _STATE:
            assert np.array_equal(sa[k], sb[k]), (t, k)
        # the twin took the same step
        assert torch.equal(ra, rz) and torch.equal(ta, tz) and torch.equal(ua, uz), t
        done = ((ta | ua) != 0).cpu().numpy()
        stepped = mask.cpu().numpy().astype(bool) if masked else np.ones(E, dtype=bool)
        fin_h, oz_h = fin.cpu().numpy(), oz.cpu().numpy()
        fin_rows = done & stepped
        assert np.array_equal(fin_h[fin_rows], oz_h[fin_rows]), t
        assert np.isnan(fin_h[~fin_rows]).all(), t
        te, tr = ta.cpu().numpy().astype(bool), ua.cpu().numpy().astype(bool)
        counts["term"] += int((te & ~tr & stepped).sum())
        counts["trunc"] += int((tr & ~te & stepped).sum())
        counts["both"] += int((te & tr & stepped).sum())
    print(counts)
    assert counts["term"] > 0 and counts["trunc"] > 0 and counts["both"] > 0
    for h in (A, B, Z):
        h.close()


@pytest.mark.parametrize("real64", [False, True])
def test_without_autoreset_final_obs_is_obs(highway_config, real64):
    E = 64
    cfg = _cfg(highway_config, "shuffled", False, duration=2)
    env = _vec(cfg, E, _spec(cfg, "rope"), False, real64)
    env.reset(3)
    rng = np.random.default_rng(2)
    seen = 0
    for _ in range(3):
        fin = torch.full((E, env.N, env.F_out), float("nan"), device="cuda:0")
        o, _, te, tr = env.step(torch.from_numpy(_actions(rng, E, False)).cuda(), final_obs_out=fin)
        done = ((te | tr) != 0).cpu().numpy()
        seen += int(done.sum())
        assert torch.equal(fin[torch.from_numpy(done).cuda()], o[torch.from_numpy(done).cuda()])
        assert torch.isnan(fin[torch.from_numpy(~done).cuda()]).all()
    assert seen > 0
    env.close()


def test_step_final_rejects_aliased_output(highway_config):
    from highway_rope_ppo_b200 import _lib

    env = _vec(_cfg(highway_config, "sorted", False), 8, None, True, False)
    a = torch.zeros((8, 2), device="cuda:0")
    with pytest.raises(ValueError):
        env.step(a, final_obs_out=torch.zeros(3, device="cuda:0"))
    with pytest.raises(_lib.HrpError, match="final_obs"):
        env.step(a, final_obs_out=env.obs)
    env.close()


# ------------------------------------------------------------------------------------------------ hrp_gae_ex
def _gae_ex(lib, r, v, te, tr, fv, lv, T, E, gamma=0.99, lam=0.95):
    adv = torch.empty((T, E), device="cuda:0")
    ret = torch.empty((T, E), device="cuda:0")
    from highway_rope_ppo_b200 import _lib

    _lib.check(lib.hrp_gae_ex(r.data_ptr(), v.data_ptr(), te.data_ptr(), tr.data_ptr(), _lib.ptr(fv), _lib.ptr(lv), T, E,
                              gamma, lam, adv.data_ptr(), ret.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "hrp_gae_ex")
    return adv, ret


def _gae(lib, r, v, d, lv, T, E, gamma=0.99, lam=0.95):
    adv = torch.empty((T, E), device="cuda:0")
    ret = torch.empty((T, E), device="cuda:0")
    from highway_rope_ppo_b200 import _lib

    _lib.check(lib.hrp_gae(r.data_ptr(), v.data_ptr(), d.data_ptr(), _lib.ptr(lv), T, E, gamma, lam, adv.data_ptr(),
                           ret.data_ptr(), torch.cuda.current_stream().cuda_stream), "hrp_gae")
    return adv, ret


@pytest.mark.parametrize("T", [1, 50, 2048])
@pytest.mark.parametrize("with_last", [True, False])
def test_gae_ex_matches_oracle_and_gae(T, with_last):
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    E = 4096
    rng = np.random.default_rng(T)
    r = rng.normal(size=(T, E)).astype(np.float32)
    v = rng.normal(size=(T, E)).astype(np.float32)
    te = rng.random((T, E)) < 0.05
    tr = rng.random((T, E)) < 0.08          # some steps both: terminated wins
    fv = rng.normal(size=(T, E)).astype(np.float32)
    fv[~(tr & ~te)] = np.nan               # the rows hrp_gae_ex must not read
    lv = rng.normal(size=E).astype(np.float32) if with_last else None
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    u8 = lambda x: d(x.astype(np.uint8))
    adv, ret = _gae_ex(lib, d(r), d(v), u8(te), u8(tr), d(fv), None if lv is None else d(lv), T, E)
    want_a, want_r = gb.gae(r, v, te, tr, fv, 0.0 if lv is None else lv)
    adv, ret = adv.cpu().numpy(), ret.cpu().numpy()
    assert np.isfinite(adv).all()
    np.testing.assert_allclose(adv, want_a, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(ret, want_r, rtol=1e-6, atol=1e-6)
    print(f"T={T}: {np.mean(adv == want_a):.6f} of the advantages bit-equal to the fp64 oracle")
    # nothing truncated, or no final_value: bit-identical to hrp_gae on done = terminated | truncated
    ga, gr = _gae(lib, d(r), d(v), u8(te | tr), None if lv is None else d(lv), T, E)
    xa, xr = _gae_ex(lib, d(r), d(v), u8(te), u8(tr), None, None if lv is None else d(lv), T, E)
    assert torch.equal(xa, ga) and torch.equal(xr, gr)
    none = np.zeros_like(tr)
    ga, gr = _gae(lib, d(r), d(v), u8(te), None if lv is None else d(lv), T, E)
    xa, xr = _gae_ex(lib, d(r), d(v), u8(te), u8(none), d(fv), None if lv is None else d(lv), T, E)
    assert torch.equal(xa, ga) and torch.equal(xr, gr)


# ------------------------------------------------------------------------------------------------ rollout
def _setup(highway_config, discrete, E, seed=7):
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_vec_env
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    torch.manual_seed(4)
    np.random.seed(4)
    cfg = _cfg(highway_config, "sorted", discrete, duration=6)
    env = make_vec_env(Condition.SORTED, cfg, num_envs=E, seed=seed)
    S = env.N * env.F_out
    agent = PPOAgent(S, 5 if discrete else 2, hidden_dim=64, batch_size=256, epochs=1, discrete=discrete)
    return env, agent, env.reset(seed).clone()


class _Recorder:
    """Wraps ppo.agent.gae to record the advantages the update used and how they were asked for."""

    def __init__(self, monkeypatch):
        from highway_rope_ppo_b200.ppo import agent as mod

        self.calls = []
        real = mod.gae

        def wrapped(*a, **kw):
            out = real(*a, **kw)
            self.calls.append(({k: (v.clone() if torch.is_tensor(v) else v) for k, v in kw.items()}, out[0].clone()))
            return out

        monkeypatch.setattr(mod, "gae", wrapped)


@pytest.mark.parametrize("discrete", [False, True], ids=["gaussian", "categorical-meta"])
def test_bootstrapped_rollout(highway_config, discrete, monkeypatch):
    from highway_rope_ppo_b200.training.routine import collect_rollout

    E, T, R = 256, 8, 3
    runs = {}
    for name, boot, use_graph in (("eager", True, False), ("graph", True, True), ("plain", False, True)):
        env, agent, obs = _setup(highway_config, discrete, E)
        rec = _Recorder(monkeypatch)
        got = []
        for it in range(R):
            r = collect_rollout(env, agent, T, obs, use_graph=use_graph, bootstrap_truncated=boot)
            snap = {k: v.clone() for k, v in r.items()}
            if boot:
                # final_value is the critic of final_states, with the parameters of this rollout
                tr = (r["truncated"] != 0) & (r["terminated"] == 0)
                _, _, fv = agent.actor_critic.forward(r["final_states"].reshape(T * E, -1))
                assert tr.any()
                assert torch.equal(fv.view(T, E)[tr], r["final_value"][tr]), it
            obs = r["states"][T].clone()
            _, _, lv = agent.actor_critic.forward(obs.view(E, -1))
            agent.update(last_value=lv.view(-1))
            kw, adv = rec.calls[-1]
            assert ("final_value" in kw) == boot
            want, _ = gb.gae(snap["reward"].cpu().numpy(), snap["value"].cpu().numpy(), snap["terminated"].cpu().numpy(),
                             snap["truncated"].cpu().numpy(), snap["final_value"].cpu().numpy() if boot else None,
                             lv.view(-1).cpu().numpy(), agent.gamma, agent.lam)
            np.testing.assert_allclose(adv.cpu().numpy(), want, rtol=1e-6, atol=1e-6)
            got.append(snap)
        runs[name] = got
        env.close()
    # graph replay == eager, every buffer.  Rows of final_states / final_value that the step does not define (envs
    # that did not finish) hold what the buffers held before: zeros in the eager run, which allocates per rollout,
    # the previous rollout's in the graph run, which reuses the captured buffers.
    for a, b in zip(runs["eager"], runs["graph"]):
        assert a.keys() == b.keys()
        done = (a["terminated"] | a["truncated"]) != 0
        tr = (a["truncated"] != 0) & (a["terminated"] == 0)
        for k in a:
            if k == "final_states":
                assert torch.equal(a[k][done], b[k][done]), k
            elif k == "final_value":
                assert torch.equal(a[k][tr], b[k][tr]), k
            else:
                assert torch.equal(a[k], b[k]), k
    # the flag changes no state, action, reward or flag of the first rollout (the updates then differ)
    a, b = runs["graph"][0], runs["plain"][0]
    assert "final_states" not in b
    for k in b:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("discrete", [False, True], ids=["gaussian", "categorical-meta"])
def test_plain_rollout_after_bootstrapped_one_has_reference_semantics(highway_config, discrete, monkeypatch):
    from highway_rope_ppo_b200.training.routine import collect_rollout, rollout_and_update

    E, T = 256, 8
    env, agent, obs = _setup(highway_config, discrete, E)
    rec = _Recorder(monkeypatch)
    _, obs = rollout_and_update(env, agent, T, obs, bootstrap_truncated=True)
    assert "final_value" in rec.calls[-1][0]
    # into the same buffers, without an update in between
    r = collect_rollout(env, agent, T, obs, bootstrap_truncated=True)
    r2 = collect_rollout(env, agent, T, r["states"][T].clone())
    assert r2 is r and "final_value" in r2   # the buffers are reused, the stale final values stay ...
    assert ((r2["truncated"] != 0) & (r2["terminated"] == 0)).any()
    snap = {k: v.clone() for k, v in r2.items()}
    agent.update(last_value=0.0)
    kw, adv = rec.calls[-1]
    assert "final_value" not in kw          # ... and are not used
    want = np.stack([ppo_ref.gae(snap["reward"][:, e].cpu().numpy(), snap["value"][:, e].cpu().numpy(),
                                 snap["done"][:, e].cpu().numpy(), 0.0, agent.gamma, agent.lam)[0] for e in range(E)], 1)
    np.testing.assert_allclose(adv.cpu().numpy(), want, rtol=1e-6, atol=1e-6)
    env.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_bootstrapped_update_keeps_ranks_bit_identical():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29643", os.path.join(root, "tools", "p2p_check.py"), "--bootstrap-truncated"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "bootstrapped truncation" in res.stdout and "identical on every rank: True" in res.stdout, res.stdout[-3000:]
