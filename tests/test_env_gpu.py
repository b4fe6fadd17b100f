"""GPU parity of the simulator kernels (hrp_env_step / observe / reset through the C-ABI) against the
CPU oracle (oracle/highway_oracle.c).  Three kinds of comparison, none of which waives an env-step:

1. STATE INJECTION, fp32 product kernel, either-branch rule.  Every step the oracle's fp64 state is injected
   into the GPU handle, both sides step once on the same action and everything is compared: lane and
   target-lane indices, crashed / pending-impact flags, terminated / truncated and the vehicle index shown in
   every observation row EXACTLY; x, y: 1e-3 m; speed: 2e-4 m/s; heading: 1e-4 rad; reward: 2e-5; observation
   entries: 2e-5 (normalised units); IDM timer: 1e-9.  The kernel integrates in fp32 (x and the lane-change
   timer in fp64), so a decision the oracle takes within MARGIN = 1e-3 of its threshold may legitimately fall
   the other way.  Such a step is NOT skipped: the oracle is re-run from the same state with its marginal
   decisions forced the other way (keyed decisions, highway_oracle.h), breadth first over combinations, and the
   kernel must equal ONE of the outcomes in full.  Counts are reported as agree / flipped / neither and any
   `neither` fails the test.  Vehicles that act below 0.5 m/s (the steering controller divides by the speed
   twice, and IDM vehicles reversing in a jam have an unstable lateral loop: rounding is amplified by > 1e3 in
   one step) get their continuous tolerances widened by 1e3, vehicles within 60 m of one by 30 (oracle/parity.py);
   nothing discrete is relaxed for them.
2. STATE INJECTION and FREE RUNNING, fp64 validation instantiation of the same kernels (HRP_ENV_REAL64): with
   no rounding in the way the discrete state must be bit-exact on 100 % of the steps -- the margin rule shrinks to
   exact ties (1e-9; in practice the contact tests of crashed vehicles resting against each other, whose
   separations are 0 to 1e-13 m, a handful per 10 000 steps) -- and the continuous state within 1e-7 (positions and impacts 2e-6: separating-axis ties between nearly parallel
   rectangles, oracle/parity.py); free running means ONE injection followed by 45 steps of both sides with
   in-kernel respawn, which exercises what per-step injection hides (pending impacts crossing a step boundary,
   episode / draw counters, accumulated state).
3. FREE-RUNNING WINDOWS of the fp32 kernel: inject once, run 5 / 15 / 40 steps on both sides, compare every step
   until the first step on which the oracle reports a decision closer than the accumulated drift allows.
"""
import copy
from collections import Counter

import numpy as np
import pytest
import torch

from oracle import highway as oh

pytestmark = pytest.mark.gpu

from oracle.parity import DISCRETE, MARGIN, MARGIN64, SLOW_FACTOR, TOL, TOL64, Got as _Got, either_branch as _either_branch, \
    frame_search as _frame_search, mismatch as _mismatch


def _vec(cfg, E, **kw):
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv

    return HighwayVecEnv(cfg, E, device="cuda:0", **kw)


def _stack_states(envs):
    sts = [e.get_state() for e in envs]
    out = {k: np.stack([s[k] for s in sts]) for k in oh.STATE_F64 + oh.STATE_I32}
    out["time"] = np.array([s["time"] for s in sts])
    return out


def _cfg(base, **over):
    c = copy.deepcopy(base)
    for k, v in over.items():
        if isinstance(v, dict):
            c[k].update(v)
        else:
            c[k] = v
    return c


def test_philox_matches_oracle():
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(0)
    for _ in range(64):
        ctr = rng.integers(0, 2**32, 4, dtype=np.uint64).astype(np.uint32)
        key = rng.integers(0, 2**32, 2, dtype=np.uint64).astype(np.uint32)
        out = np.zeros(4, dtype=np.uint32)
        lib.hrp_philox4x32_10(ctr.ctypes.data, key.ctypes.data, out.ctypes.data)
        assert np.array_equal(out, oh.philox4x32_10(ctr, key))


@pytest.mark.parametrize("real64", [False, True])
@pytest.mark.parametrize("seed,base", [(0, 0), (42, 0), (2**40 + 7, 1000)])
def test_reset_matches_oracle(highway_config, seed, base, real64):
    E = 96
    env = _vec(highway_config, E, env_id_base=base, real64=real64)
    env.reset(seed)
    st = env.get_state()
    o = oh.OracleEnv(highway_config)
    for e in range(E):
        o.reset(seed, env_id=base + e, episode=0)
        ref = o.get_state()
        for k in DISCRETE:
            assert np.array_equal(st[k][e], ref[k]), k
        np.testing.assert_allclose(st["x"][e], ref["x"], atol=1e-9)
        np.testing.assert_allclose(st["timer"][e], ref["timer"], atol=1e-8)
        for k in ("y", "speed", "target_speed", "delta", "heading"):
            np.testing.assert_allclose(st[k][e], ref[k], rtol=1e-12 if real64 else 2e-7, atol=1e-7, err_msg=k)
        assert st["time"][e] == 0.0 and st["episode"][e] == 0
    env.close()


def _injected_parity(cfg, E, steps, seed, action_fn, sorted_obs=True, obs_tol=2e-5, real64=False, embed=None):
    """State-injection parity.  Returns a dict: agree / flipped / neither env-step counts, the kinds of the decisions
    that had to be flipped, the worst continuous errors of the agreeing steps and the first few failures.  With an
    EmbedSpec `embed`, a second handle with that fused embedding is injected and stepped alongside: "embedded" lists
    (plain observation, fused observation) per step."""
    N = cfg["observation"]["vehicles_count"]
    env = _vec(cfg, E, autoreset=False, real64=real64)
    fused = None if embed is None else _vec(cfg, E, autoreset=False, real64=real64, embed=embed)
    ktrace = env.enable_trace()   # per-frame snapshots, for the frame-by-frame search
    oracles = [oh.OracleEnv(cfg) for _ in range(E)]
    for e, o in enumerate(oracles):
        o.reset(seed, env_id=e, episode=0)
    rng = np.random.default_rng(seed)
    rows = torch.zeros((E, N), dtype=torch.int32, device="cuda:0")
    tol, rew_tol = (TOL64, 1e-6) if real64 else (TOL, 2e-5)
    obs_tol = 1e-6 if real64 else obs_tol
    stats = {"agree": 0, "flipped": 0, "neither": 0, "kinds": Counter(), "worst": {}, "failures": [], "by_frames": 0,
             "embedded": []}
    for t in range(steps):
        sts = [o.get_state() for o in oracles]
        st = {k: np.stack([s[k] for s in sts]) for k in oh.STATE_F64 + oh.STATE_I32}
        st["time"] = np.array([s["time"] for s in sts])
        env.set_state(st)
        actions = action_fn(rng, E, t).astype(np.float32)
        perm = None
        if not sorted_obs:
            perm = np.stack([rng.permutation(N - 1) for _ in range(E)]).astype(np.int32)
        obs, rew, term, trunc = env.step(torch.from_numpy(actions).cuda(),
                                         perm=None if perm is None else torch.from_numpy(perm).cuda(),
                                         row_vehicle=rows)
        state = env.get_state()
        obs, rew, term, trunc, rv = (x.cpu().numpy() for x in (obs, rew, term, trunc, rows))
        if fused is not None:
            fused.set_state(st)
            fo = fused.step(torch.from_numpy(actions).cuda(), perm=None if perm is None else torch.from_numpy(perm).cuda())[0]
            stats["embedded"].append((obs, fo.cpu().numpy()))
        trace_host = None
        for e, o in enumerate(oracles):
            got = _Got(state, e, obs, rew, term, trunc, rv)
            pe = None if perm is None else perm[e]
            r, te, tr = o.step(actions[e])
            want_obs, want_rows = o.observe(perm=pe, with_rows=True)
            why = _mismatch(got, o, r, te, tr, want_obs, want_rows, tol, obs_tol, rew_tol, stats["worst"])
            if why is None:
                stats["agree"] += 1
            else:
                # fp64 kernel: only exact ties may be flipped (margins below 1e-9: resting contacts of a pile-up)
                mg = MARGIN64 if real64 else MARGIN
                forced = _either_branch(o, sts[e], actions[e], pe, got, tol, obs_tol, rew_tol, why=why, margin=mg)
                if not forced:
                    # a chain of exactly-touching contacts (pile-up): follow the kernel's per-frame trace
                    if trace_host is None:
                        trace_host = ktrace.cpu().numpy()
                    ttol = np.array([tol[k] for k in ("x", "y", "speed", "heading", "impact_x", "impact_y")])
                    forced = _frame_search(o, sts[e], actions[e], pe, got, trace_host[e], tol, obs_tol, rew_tol, margin=mg,
                                           trace_tol=ttol)
                    stats["by_frames"] += 1 if forced else 0
                if forced:
                    stats["flipped"] += 1
                    stats["kinds"].update(oh.decode_key(k).split("[")[0] for k in forced)
                else:
                    stats["neither"] += 1
                    if len(stats["failures"]) < 5:
                        stats["failures"].append((t, e, why))
            if te or tr:  # reference loop: reset right after done
                o.reset(seed, env_id=e, episode=1 + t)
    env.close()
    if fused is not None:
        fused.close()
    return stats


def _report(name, s):
    n = s["agree"] + s["flipped"] + s["neither"]
    print(f"{name}: {n} env-steps: agree {s['agree']}, flipped {s['flipped']} {dict(s['kinds'])} ({s['by_frames']} by the "
          f"frame-by-frame search), neither {s['neither']}; "
          f"max abs err {({k: float(f'{v:.3g}') for k, v in s['worst'].items()})}")
    assert s["neither"] == 0, s["failures"]
    return n


def _random_actions(rng, E, t):
    return rng.uniform(-1, 1, (E, 2))


def _gentle_actions(rng, E, t):
    a = rng.uniform(-1, 1, (E, 2))
    a[:, 1] *= 0.08  # small steering: long episodes in traffic, lane changes of the IDM vehicles dominate
    return a


def test_step_parity_random_actions(highway_config):
    """>= 1000 injected-state env-steps with uniformly random actions (crashes, off-road, respawns)."""
    s = _injected_parity(highway_config, E=48, steps=25, seed=1, action_fn=_random_actions)
    assert _report("random actions", s) >= 1000 and s["flipped"] <= 0.3 * s["agree"]


def test_step_parity_gentle_actions(highway_config):
    """Long episodes (40 steps, truncation) where IDM / MOBIL traffic interaction is the bulk of the work."""
    s = _injected_parity(highway_config, E=32, steps=42, seed=2, action_fn=_gentle_actions)
    assert _report("gentle actions", s) >= 1000 and s["flipped"] <= 0.3 * s["agree"]


def test_step_parity_shuffled_30_rows_7_features(highway_config):
    """BASELINE config 3 shape: N = 30 observed vehicles, all 7 features, shuffled with an injected permutation."""
    cfg = _cfg(highway_config, observation=dict(vehicles_count=30, order="shuffled",
                                               features=["presence", "x", "y", "vx", "vy", "cos_h", "sin_h"]))
    s = _injected_parity(cfg, E=16, steps=20, seed=3, action_fn=_random_actions, sorted_obs=False)
    assert _report("shuffled N=30 F=7", s) >= 320


def test_step_parity_dense_small_road(highway_config):
    """Edge sizes: 2 lanes, 12 vehicles at density 3 (frequent contacts), 5 observed rows, see_behind."""
    cfg = _cfg(highway_config, lanes_count=2, vehicles_count=12, vehicles_density=3,
               observation=dict(vehicles_count=5, see_behind=True))
    s = _injected_parity(cfg, E=32, steps=30, seed=4, action_fn=_random_actions)
    assert _report("dense 2-lane", s) >= 960


def _meta_actions(rng, E, t):
    a = np.zeros((E, 2))
    a[:, 0] = rng.integers(0, 5, E)
    return a


def _meta_cfg(highway_config):
    cfg = _cfg(highway_config)
    cfg["action"] = {"type": "DiscreteMetaAction"}
    return cfg


def test_step_parity_meta_action_ego(highway_config):
    """DiscreteMetaAction / MDPVehicle ego (north_star; unreachable through the reference runner, SURVEY F2)."""
    s = _injected_parity(_meta_cfg(highway_config), E=24, steps=40, seed=5, action_fn=_meta_actions)
    assert _report("meta-action ego", s) >= 960


def test_single_vehicle_and_max_vehicles(highway_config):
    """Edge sizes: an empty road (ego only: every observation row but the first is padding) and V = 64."""
    for vc in (0, 63):
        cfg = _cfg(highway_config, vehicles_count=vc)
        s = _injected_parity(cfg, E=8, steps=12, seed=6 + vc, action_fn=_gentle_actions)
        assert _report(f"vehicles_count {vc}", s) == 96


# ---- fp64 validation instantiation: bit-exact discrete state on every step, no margin rule -------------------------
@pytest.mark.parametrize("name", ["random", "gentle", "dense", "meta", "shuffled30"])
def test_fp64_kernel_is_exact_on_every_step(highway_config, name):
    cfg, fn, sorted_obs, E, steps = {
        "random": (highway_config, _random_actions, True, 32, 25),
        "gentle": (highway_config, _gentle_actions, True, 24, 42),
        "dense": (_cfg(highway_config, lanes_count=2, vehicles_count=12, vehicles_density=3,
                       observation=dict(vehicles_count=5, see_behind=True)), _random_actions, True, 32, 30),
        "meta": (_meta_cfg(highway_config), _meta_actions, True, 24, 40),
        "shuffled30": (_cfg(highway_config, observation=dict(vehicles_count=30, order="shuffled",
                                                             features=["presence", "x", "y", "vx", "vy", "cos_h", "sin_h"])),
                       _random_actions, False, 16, 20),
    }[name]
    s = _injected_parity(cfg, E=E, steps=steps, seed=11, action_fn=fn, sorted_obs=sorted_obs, real64=True)
    n = _report(f"fp64 kernel, {name}", s)
    # every step bit-exact in the discrete state; the only decisions that may fall the other way are exact ties
    # (margin < 1e-9: two crashed vehicles resting against each other), and they are rare
    assert n == E * steps and s["flipped"] <= 0.002 * n and set(s["kinds"]) <= {"sat_will", "sat_now", "sat_axis"}


def _free_run(cfg, E, steps, seed, action_fn, real64, window=None):
    """ONE injection (the oracle's spawn), then `steps` steps of both sides without re-injection, in-kernel respawn
    on, the oracle respawning the same episodes.  fp64 kernel: everything is compared on every step.  fp32 kernel:
    an env is compared until the first step on which the oracle took a decision by less than the drift bound."""
    N = cfg["observation"]["vehicles_count"]
    env = _vec(cfg, E, autoreset=True, real64=real64, seed=seed)
    env.reset(seed)
    oracles = [oh.OracleEnv(cfg) for _ in range(E)]
    episode = [0] * E
    for e, o in enumerate(oracles):
        o.reset(seed, env_id=e, episode=0)
    st = _stack_states(oracles)
    full = dict(st)
    state0 = env.get_state()
    full["episode"], full["obs_draw"] = state0["episode"], state0["obs_draw"]
    env.set_state(full)
    rng = np.random.default_rng(seed)
    rows = torch.zeros((E, N), dtype=torch.int32, device="cuda:0")
    live = np.ones(E, dtype=bool)
    _free_run.ended = 0
    ever_slow = np.zeros(E, dtype=bool)
    closest = np.full(E, np.inf)
    compared, lengths, worst = 0, [], {}
    for t in range(steps):
        actions = action_fn(rng, E, t).astype(np.float32)
        obs, rew, term, trunc = env.step(torch.from_numpy(actions).cuda(), row_vehicle=rows)
        state = env.get_state()
        obs, rew, term, trunc, rv = (x.cpu().numpy() for x in (obs, rew, term, trunc, rows))
        for e, o in enumerate(oracles):
            if not live[e]:
                continue
            r, te, tr = o.step(actions[e])
            margin = o.min_margin()
            if te or tr:  # the kernel respawned inside the step: the state and the observation are the new episode's
                episode[e] += 1
                o.reset(seed, env_id=e, episode=episode[e])
            want_obs, want_rows = o.observe(with_rows=True)
            margin = min(margin, o.min_margin())
            got = _Got(state, e, obs, rew, term, trunc, rv)
            if real64:
                # Discrete state, flags, rows, episode counters exact and continuous state within 1e-7 on every step.
                # A difference ends the env's window -- instead of failing -- only if the oracle itself says why the two
                # sides may have separated: (a) an exact tie (a decision margin below 1e-9: resting contacts of a
                # pile-up, the cases the injected runs resolve by flipping the tie), or (b) a vehicle of the env has
                # crawled or reversed at this or an earlier step of the window: such a vehicle is laterally UNSTABLE
                # under highway-env's own steering law, a rounding-level difference grows 5 to 8 times per simulation
                # frame for as long as it reverses (profiles/r02_reversing_vehicle_trace.txt), in the oracle as in the
                # kernel, and without re-injection nothing bounds it.  `_free_run.ended` counts those windows; the
                # injected runs check exactly those steps one at a time.
                ever_slow[e] |= bool(o.slow_vehicles().any())
                why = _mismatch(got, o, r, te, tr, want_obs, want_rows, TOL64, 1e-6, 1e-6, worst)
                if why is not None and (ever_slow[e] or margin < MARGIN64):
                    live[e] = False
                    _free_run.ended += 1
                    lengths.append(t)
                    continue
                assert why is None, (t, e, why, margin)
                assert state["episode"][e] == episode[e]
            else:
                # tolerances and the decision margin grow with the steps since the injection.  A window ends at the
                # first difference, and a difference is only legitimate if the oracle has taken a decision inside the
                # drift-scaled margin at this or an earlier step of the window (the two sides may then have branched).
                drift = 1.0 + t
                closest[e] = min(closest[e], margin / drift)
                why = _mismatch(got, o, r, te, tr, want_obs, want_rows, {k: v * drift for k, v in TOL.items()},
                                2e-5 * drift, 2e-5 * drift, worst)
                if why is not None:
                    assert closest[e] < MARGIN, (t, e, why, closest[e])
                    live[e] = False
                    lengths.append(t)
                    continue
            compared += 1
    lengths += [steps] * int(live.sum())
    env.close()
    return compared, lengths, worst


def test_fp64_kernel_free_running_45_steps(highway_config):
    """Inject once, then 45 free-running steps with in-kernel respawn: bit-exact discrete state throughout."""
    compared, _, worst = _free_run(highway_config, E=24, steps=45, seed=21, action_fn=_gentle_actions, real64=True)
    print("fp64 free run, gentle:", compared, "env-steps, max abs err", worst)
    assert compared == 24 * 45
    compared, _, worst = _free_run(highway_config, E=24, steps=30, seed=22, action_fn=_random_actions, real64=True)
    print("fp64 free run, random:", compared, "env-steps, max abs err", worst)
    assert compared == 24 * 30
    cfg = _meta_cfg(highway_config)
    compared, _, worst = _free_run(cfg, E=16, steps=45, seed=23, action_fn=_meta_actions, real64=True)
    print("fp64 free run, meta-action:", compared, "env-steps, max abs err", worst)
    assert compared == 16 * 45


@pytest.mark.parametrize("window", [5, 15, 40])
def test_fp32_kernel_free_running_windows(highway_config, window):
    """Inject once, run `window` steps on both sides, compare every step until the first marginal decision."""
    compared, lengths, worst = _free_run(highway_config, E=48, steps=window, seed=30 + window,
                                         action_fn=_gentle_actions, real64=False)
    print(f"fp32 free run, window {window}: {compared} env-steps compared, mean compared length "
          f"{np.mean(lengths):.1f}, full windows {sum(l == window for l in lengths)}/48, max abs err", worst)
    assert np.mean(lengths) >= 0.6 * window


def test_fp32_kernel_matches_fp64_kernel(highway_config):
    """The product kernel against the validation instantiation on identical injected states (no oracle involved):
    discrete state equal wherever the fp64 kernel's neighbours in state space agree, continuous state within TOL."""
    E, seed = 64, 77
    a, b = _vec(highway_config, E, autoreset=False), _vec(highway_config, E, autoreset=False, real64=True)
    a.reset(seed)
    b.reset(seed)
    g = torch.Generator(device="cuda:0").manual_seed(3)
    same = total = 0
    for t in range(20):
        b.set_state(a.get_state())   # fp32-representable states: both start from identical values
        act = torch.rand((E, 2), generator=g, device="cuda:0") * 2 - 1
        act[:, 1] *= 0.1
        a.step(act)
        b.step(act)
        sa, sb = a.get_state(), b.get_state()
        for e in range(E):
            total += 1
            if all(np.array_equal(sa[k][e], sb[k][e]) for k in DISCRETE):
                same += 1
                for k, tol in TOL.items():
                    assert np.max(np.abs(sa[k][e] - sb[k][e])) <= tol * (SLOW_FACTOR if np.any(np.abs(sb["speed"][e]) < 0.6) else 1), (k, t, e)
    print(f"fp32 vs fp64 kernel: discrete state identical on {same}/{total} env-steps")
    assert same >= 0.8 * total
    a.close(); b.close()


def test_shuffle_draw_matches_oracle_permutation(highway_config):
    """Without an injected permutation the kernel draws it from Philox(seed, env id, draw counter)."""
    cfg = _cfg(highway_config, observation=dict(order="shuffled"))
    E, N, seed, base = 40, 15, 99, 500
    env = _vec(cfg, E, env_id_base=base, autoreset=False)
    env.reset(seed)
    rows = torch.zeros((E, N), dtype=torch.int32, device="cuda:0")
    st0 = env.get_state()
    env.observe(row_vehicle=rows)
    rv = rows.cpu().numpy()
    o = oh.OracleEnv(cfg)
    for e in range(E):
        o.reset(seed, env_id=base + e, episode=0)
        perm = oh.shuffle_perm(seed, base + e, int(st0["obs_draw"][e]), N - 1)
        _, want = o.observe(perm=perm, with_rows=True)
        assert np.array_equal(rv[e], want)
    assert np.all(env.get_state()["obs_draw"] == st0["obs_draw"] + 1)
    env.close()


def test_autoreset_respawns_inside_the_step(highway_config):
    """A finished env is respawned by the same launch: episode counter +1, time 0, fresh spawn == oracle's."""
    E, seed = 64, 7
    env = _vec(highway_config, E, autoreset=True)
    env.reset(seed)
    st = env.get_state()
    st["time"][::2] = 39.0  # every other env truncates on this step
    env.set_state(st)
    a = torch.zeros((E, 2), device="cuda:0")
    obs, rew, term, trunc = env.step(a)
    trunc = trunc.cpu().numpy().astype(bool)
    assert trunc[::2].all() and not trunc[1::2].any()
    got = env.get_state()
    o = oh.OracleEnv(highway_config)
    for e in range(0, E, 2):
        o.reset(seed, env_id=e, episode=1)
        ref = o.get_state()
        assert got["episode"][e] == 1 and got["time"][e] == 0.0
        np.testing.assert_allclose(got["x"][e], ref["x"], atol=1e-9)
        assert np.array_equal(got["lane"][e], ref["lane"])
        np.testing.assert_allclose(obs[e].cpu().numpy(), o.observe(), atol=2e-6)
    # envs that did not finish (no truncation, no crash in this step) keep their episode and advance time
    alive = ~(trunc | term.cpu().numpy().astype(bool))
    assert alive[1::2].sum() > E // 4
    assert np.all(got["episode"][alive] == 0) and np.all(got["time"][alive] == 1.0)
    assert np.all(got["episode"][~alive] == 1) and np.all(got["time"][~alive] == 0.0)
    env.close()


def test_full_size_invariants(highway_config):
    """BASELINE size (4096 envs): size-independent properties after 45 free-running steps with autoreset."""
    E = 4096
    env = _vec(highway_config, E, autoreset=True)
    env.reset(123)
    g = torch.Generator(device="cuda:0").manual_seed(42)
    ep_done = torch.zeros(E, dtype=torch.int64, device="cuda:0")
    for t in range(45):
        a = torch.rand((E, 2), generator=g, device="cuda:0") * 2 - 1
        a[:, 1] *= 0.1
        obs, rew, term, trunc = env.step(a)
        assert torch.isfinite(obs).all() and torch.isfinite(rew).all()
        assert (rew >= 0).all() and (rew <= 1.0 + 1e-6).all()
        assert (obs.abs() <= 1.0 + 1e-6).all()
        ep_done += (term | trunc).long()
    st = env.get_state()
    assert np.all(st["time"] <= 40.0) and np.all(st["time"] >= 0.0)
    assert np.all(st["episode"] == ep_done.cpu().numpy())   # every done respawned exactly once
    assert np.all((st["lane"] >= 0) & (st["lane"] < 4))
    assert np.all(np.isfinite(st["x"])) and np.all(np.isfinite(st["speed"]))
    # ego row is absolute: x / 100 clipped to 1 (a forward-driving ego is always beyond x = 100, SURVEY F6)
    o = obs.cpu().numpy()
    np.testing.assert_allclose(o[:, 0, 0], np.clip(st["x"][:, 0] / 100.0, -1, 1), atol=1e-6)
    np.testing.assert_allclose(o[:, 0, 1], np.clip(st["y"][:, 0] / 100.0, -1, 1), atol=1e-6)
    assert (o[:, 0, 0] == 1.0).mean() > 0.95
    # sorted observation: |dx| non-decreasing over the non-padding rows
    o = obs.cpu().numpy()
    dx = np.abs(o[:, 1:, 0])
    present = np.any(o[:, 1:, :] != 0, axis=-1)
    for e in range(0, E, 37):
        k = int(present[e].sum())
        assert np.all(np.diff(dx[e, :k]) >= -1e-7)
    env.close()


def test_host_buffer_entry_points_match_device_path(highway_config):
    E = 32
    a_env, b_env = _vec(highway_config, E), _vec(highway_config, E)
    obs_h = np.zeros((E, 15, 4), dtype=np.float32)
    a_env.reset_host(5, obs_h)
    obs_d = b_env.reset(5)
    assert np.array_equal(obs_h, obs_d.cpu().numpy())
    rew, te, tr = np.zeros(E, np.float32), np.zeros(E, np.uint8), np.zeros(E, np.uint8)
    rng = np.random.default_rng(0)
    for _ in range(5):
        act = rng.uniform(-1, 1, (E, 2)).astype(np.float32)
        a_env.step_host(act, obs_h, rew, te, tr)
        o, r, t1, t2 = b_env.step(torch.from_numpy(act).cuda())
        assert np.array_equal(obs_h, o.cpu().numpy()) and np.array_equal(rew, r.cpu().numpy())
        assert np.array_equal(te, t1.cpu().numpy()) and np.array_equal(tr, t2.cpu().numpy())
    # device actions on the caller's stream and page-locked result buffers (hrp_env_step_host_on): same results
    obs_p = torch.zeros((E, 15, 4)).pin_memory()
    rew_p, te_p, tr_p = torch.zeros(E).pin_memory(), torch.zeros(E, dtype=torch.uint8).pin_memory(), \
        torch.zeros(E, dtype=torch.uint8).pin_memory()
    for _ in range(5):
        act = torch.from_numpy(rng.uniform(-1, 1, (E, 2)).astype(np.float32)).cuda()
        a_env.step_host(act, obs_p.numpy(), rew_p.numpy(), te_p.numpy(), tr_p.numpy())
        o, r, t1, t2 = b_env.step(act)
        assert torch.equal(obs_p, o.cpu()) and torch.equal(rew_p, r.cpu())
        assert torch.equal(te_p.bool(), t1.cpu().bool()) and torch.equal(tr_p.bool(), t2.cpu().bool())
    with pytest.raises(ValueError):
        a_env.step_host(torch.zeros(3, device="cuda:0"), obs_h, rew, te, tr)
    a_env.close(); b_env.close()


class _KernelEnv:
    """One GPU env behind the OracleEnv interface, so that the hand-derived scenarios of tests/test_oracle_cpu.py can
    be replayed on the kernel itself (no oracle involved)."""

    def __init__(self, cfg):
        self.env = _vec(cfg, 1, autoreset=False)
        self.N = cfg["observation"]["vehicles_count"]

    def reset(self, seed):
        self.env.reset(seed)

    def get_state(self):
        st = self.env.get_state()
        out = {k: st[k][0].copy() for k in oh.STATE_F64 + oh.STATE_I32}
        out["time"] = float(st["time"][0])
        self._extra = {k: st[k] for k in ("episode", "obs_draw")}
        return out

    def set_state(self, st):
        full = {k: np.asarray(st[k])[None] for k in oh.STATE_F64 + oh.STATE_I32}
        full["time"] = np.array([st["time"]])
        full.update(self._extra)
        self.env.set_state(full)

    def step(self, action):
        obs, r, te, tr = self.env.step(torch.tensor([action], dtype=torch.float32, device="cuda:0"))
        self.obs = obs[0].cpu().numpy()
        return float(r[0]), bool(te[0]), bool(tr[0])

    def close(self):
        self.env.close()


def test_kernel_reward_extremes_by_hand(highway_config):
    """The scenario of test_oracle_cpu.test_sim_reward_extremes on the CUDA kernel (fp32: 2e-6)."""
    env = _KernelEnv(_cfg(highway_config, vehicles_count=0))
    for lane, speed, want in ((3, 30.0, 1.0), (0, 20.0, 1.0 / 1.5), (3, 35.0, 1.0), (1, 25.0, (0.1 / 3 + 0.2 + 1.0) / 1.5)):
        env.reset(1)
        st = env.get_state()
        st["x"][0], st["y"][0], st["speed"][0], st["heading"][0] = 100.0, 4.0 * lane, speed, 0.0
        st["lane"][0] = st["target_lane"][0] = lane
        env.set_state(st)
        r, term, trunc = env.step([0.0, 0.0])
        assert abs(r - want) < 2e-6 and not term and not trunc, (lane, speed, r, want)
    env.close()


def test_kernel_mobil_safety_and_timer_by_hand(highway_config):
    """MOBIL on the kernel: the unsafe lane is refused, the later candidate wins otherwise, and a timer reset to zero
    fires on the 16th frame (fp64 timer: 15 x 1/15 < 1)."""
    env = _KernelEnv(_cfg(highway_config, vehicles_count=3))
    env.reset(5)
    st = env.get_state()
    st["x"][:] = [0.0, 200.0, 235.0, 192.0]
    st["y"][:] = [12.0, 4.0, 4.0, 8.0]
    st["lane"][:] = st["target_lane"][:] = [3, 1, 1, 2]
    st["speed"][:] = [0.0, 25.0, 18.0, 30.0]
    st["target_speed"][:] = [0.0, 30.0, 18.0, 30.0]
    st["delta"][:] = 4.0
    st["timer"][:] = [0.0, 1.0 + 1e-9, 0.0, 0.0]
    st["heading"][:] = 0.0
    st["crashed"][:] = 0
    st["has_impact"][:] = 0
    env.set_state(st)
    env.step([0.0, 0.0])
    assert env.get_state()["target_lane"][1] == 0          # lane 2 would force its follower below -2 m/s^2
    st["x"][3] = 1000.0
    env.set_state(st)
    env.step([0.0, 0.0])
    assert env.get_state()["target_lane"][1] == 2          # both lanes acceptable: the later candidate overwrites
    st["timer"][1] = 0.0
    env.set_state(st)
    env.step([0.0, 0.0])
    assert env.get_state()["target_lane"][1] == 1          # 15 frames of 1/15: 1.0 < timer never true
    env.step([0.0, 0.0])
    assert env.get_state()["target_lane"][1] == 2          # fires on the first frame of the next step
    env.close()


def test_kernel_rectangle_contact_thresholds_by_hand(highway_config):
    """5 x 2 m rectangles at equal speed: contact iff both axis gaps are closed (kernel SAT, rank-neighbour search)."""
    env = _KernelEnv(_cfg(highway_config, vehicles_count=1))
    for dx, dy, hit in ((5.05, 0.0, False), (4.95, 0.0, True), (4.0, 2.05, False), (4.0, 1.95, True), (0.0, 1.99, True),
                        (6.0, 3.0, False)):
        env.reset(5)
        st = env.get_state()
        st["x"][:] = [100.0, 100.0 + dx]
        st["y"][:] = [4.0, 4.0 + dy]
        st["lane"][:] = st["target_lane"][:] = [1, 1 if dy < 2 else 2]
        st["speed"][:] = [20.0, 20.0]
        st["target_speed"][:] = [20.0, 20.0]
        st["heading"][:] = 0.0
        st["timer"][:] = 0.0
        env.set_state(st)
        r, term, trunc = env.step([0.0, 0.0])
        s1 = env.get_state()
        assert bool(s1["crashed"][0]) == hit and term == hit, (dx, dy, s1["crashed"], term)
    env.close()


def test_kernel_observation_clip_by_hand(highway_config):
    """Relative rows, / 100 and / 30 normalisation, clip to [-1, 1], vehicles more than 10 m behind dropped, padding."""
    env = _KernelEnv(_cfg(highway_config, vehicles_count=3))
    env.reset(5)
    st = env.get_state()
    st["x"][:] = [300.0, 450.0, 320.0, 280.0]
    st["y"][:] = [4.0, 8.0, 0.0, 4.0]
    st["lane"][:] = st["target_lane"][:] = [1, 2, 0, 1]
    st["speed"][:] = [25.0, 22.0, 28.0, 20.0]
    st["heading"][:] = 0.0
    env.set_state(st)
    obs = env.env.observe()[0].cpu().numpy()
    np.testing.assert_allclose(obs[0], [1.0, 0.04, 25.0 / 30.0, 0.0], atol=1e-6)
    np.testing.assert_allclose(obs[1], [0.2, -0.04, 3.0 / 30.0, 0.0], atol=1e-6)
    np.testing.assert_allclose(obs[2], [1.0, 0.04, -3.0 / 30.0, 0.0], atol=1e-6)
    assert np.all(obs[3:] == 0.0)
    env.close()


def test_async_host_step_in_two_groups_equals_one_env(highway_config):
    """hrp_env_step_host_async on two env groups / two streams (the pipelined host-buffer loop of bench.py): the groups
    own global env ids [0, 32) and [32, 64) and must reproduce a single 64-env handle; results are complete after the
    group's event."""
    E, half = 64, 32
    whole = _vec(highway_config, E)
    groups = [_vec(highway_config, half, env_id_base=g * half) for g in range(2)]
    streams = [torch.cuda.Stream(device="cuda:0") for _ in range(2)]
    events = [torch.cuda.Event() for _ in range(2)]
    pin = lambda *shape, dtype=torch.float32: torch.zeros(shape, dtype=dtype).pin_memory()
    bufs = [dict(obs=pin(half, 15, 4), rew=pin(half), te=pin(half, dtype=torch.uint8), tr=pin(half, dtype=torch.uint8))
            for _ in range(2)]
    want = whole.reset(9).cpu()
    for g in range(2):
        groups[g].reset_host(9, bufs[g]["obs"].numpy())
        assert torch.equal(bufs[g]["obs"], want[g * half:(g + 1) * half])
    gen = torch.Generator(device="cuda:0").manual_seed(4)
    for t in range(6):
        act = torch.rand((E, 2), generator=gen, device="cuda:0") * 2 - 1
        o, r, te, tr = whole.step(act)
        torch.cuda.synchronize()
        for g in range(2):
            with torch.cuda.stream(streams[g]):
                b = bufs[g]
                groups[g].step_host_async(act[g * half:(g + 1) * half], b["obs"].numpy(), b["rew"].numpy(), b["te"].numpy(),
                                          b["tr"].numpy())
                events[g].record()
        for g in range(2):
            events[g].synchronize()
            sl = slice(g * half, (g + 1) * half)
            assert torch.equal(bufs[g]["obs"], o[sl].cpu()) and torch.equal(bufs[g]["rew"], r[sl].cpu()), (t, g)
            assert torch.equal(bufs[g]["te"], te[sl].cpu()) and torch.equal(bufs[g]["tr"], tr[sl].cpu())
    with pytest.raises(Exception):   # pageable buffers cannot complete after the call returns
        groups[0].step_host_async(act[:half], np.zeros((half, 15, 4), np.float32), np.zeros(half, np.float32),
                                  np.zeros(half, np.uint8), np.zeros(half, np.uint8))
    whole.close()
    for g in groups:
        g.close()


def test_per_env_seeds_and_step_mask_reproduce_single_env_handles(highway_config):
    """hrp_env_set_seeds / hrp_env_set_step_mask (the multiplexed sweep, experiments/multiplex.py): env e of a shared
    handle, seeded with seeds[e] and stepped only when mask[e], is bit for bit the single-env handle of a run that
    called reset(seed=seeds[e]) -- state, observation, reward, flags and the shuffle draws -- while its neighbours are
    reset and stepped on their own schedules."""
    cfg = _cfg(highway_config, observation=dict(order="shuffled"))
    R, T = 5, 12
    seeds = [42, 1042, 7, 2**40 + 3, 99]
    rng = np.random.default_rng(3)
    actions = rng.uniform(-1, 1, (T, R, 2)).astype(np.float32)
    active = rng.random((T, R)) < 0.7
    active[0] = True
    resets = {(4, 1): 555, (7, 3): 556}          # (t, env) -> new seed: a run starts another episode
    # reference: R single-env handles driven one by one
    want = []
    singles = [_vec(cfg, 1, autoreset=False) for _ in range(R)]
    for e, env in enumerate(singles):
        env.reset(seeds[e])
    for t in range(T):
        row = []
        for e, env in enumerate(singles):
            if (t, e) in resets:
                env.reset(resets[(t, e)])
            if active[t, e]:
                o, r, te, tr = env.step(torch.from_numpy(actions[t, e:e + 1]).cuda())
                row.append((o.cpu().numpy()[0].copy(), float(r[0]), int(te[0]), int(tr[0])))
            else:
                row.append(None)
        want.append(row)
    want_state = [env.get_state() for env in singles]
    for env in singles:
        env.close()
    # one shared handle
    env = _vec(cfg, R, autoreset=False)
    sd = torch.tensor(seeds, dtype=torch.int64, device="cuda:0")
    mask = torch.zeros(R, dtype=torch.uint8, device="cuda:0")
    env.set_env_seeds(sd)
    env.set_step_mask(mask)
    env.reset()
    for t in range(T):
        for (tt, e), s in resets.items():
            if tt == t:
                sd[e] = s
                m = torch.zeros(R, dtype=torch.uint8, device="cuda:0")
                m[e] = 1
                env.reset(mask=m)
        mask.copy_(torch.from_numpy(active[t].astype(np.uint8)))
        o, r, te, tr = env.step(torch.from_numpy(actions[t]).cuda())
        o, r, te, tr = o.cpu().numpy(), r.cpu().numpy(), te.cpu().numpy(), tr.cpu().numpy()
        for e in range(R):
            if want[t][e] is not None:
                wo, wr, wte, wtr = want[t][e]
                assert np.array_equal(o[e], wo) and float(r[e]) == wr and int(te[e]) == wte and int(tr[e]) == wtr, (t, e)
    got = env.get_state()
    for e in range(R):
        for k in oh.STATE_F64 + oh.STATE_I32:
            assert np.array_equal(got[k][e], want_state[e][k][0]), (e, k)
    env.close()
