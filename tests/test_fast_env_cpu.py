"""highway-fast-v0, CPU side: the gym_id config key and its defaults, the C ABI field that selects the collision rule,
and the fp64 oracle's ego-only collision rule (tests/fast_oracle.py) against cases worked out by hand (DESIGN.md
Appendix C)."""
import copy
import ctypes as C

import numpy as np
import pytest

from fast_oracle import FAST, highway as fast_oh, oracle_module
from oracle import highway as oh

KINEMATICS = {"type": "Kinematics", "vehicles_count": 5, "features": ["presence", "x", "y", "vx", "vy"]}


def test_resolve_config_applies_the_fast_defaults():
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg, resolve_config

    full = resolve_config({"gym_id": FAST})
    assert full["gym_id"] == FAST
    assert (full["simulation_frequency"], full["lanes_count"], full["vehicles_count"], full["duration"],
            full["ego_spacing"]) == (5, 3, 20, 30, 1.5)
    assert full["policy_frequency"] == 1 and full["vehicles_density"] == 1   # the rest is HighwayEnv's
    c = build_cfg({"gym_id": FAST})
    assert (c.simulation_frequency, c.lanes_count, c.vehicles_count, c.duration, c.ego_spacing) == (5, 3, 20, 30.0, 1.5)
    assert c.ego_collisions_only == 1 and c.obs_vehicles == 5 and c.ego_mode == 1


def test_user_keys_win_over_the_fast_defaults():
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    c = build_cfg({"gym_id": FAST, "lanes_count": 5, "ego_spacing": 3, "duration": 12})
    assert (c.lanes_count, c.ego_spacing, c.duration) == (5, 3.0, 12.0)
    assert (c.simulation_frequency, c.vehicles_count) == (5, 20) and c.ego_collisions_only == 1


def test_reference_config_on_the_fast_id(highway_config):
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    v0 = build_cfg(highway_config)
    fast = build_cfg(dict(highway_config, gym_id=FAST))
    assert (fast.simulation_frequency, fast.vehicles_count + 1, fast.lanes_count, fast.duration) == (15, 51, 4, 40.0)
    assert fast.ego_spacing == 1.5 and fast.ego_collisions_only == 1
    assert v0.ego_spacing == 2.0 and v0.ego_collisions_only == 0
    # the two differ in ego spacing and in the collision rule only
    as_list = lambda v: list(v) if hasattr(v, "__len__") else v
    diff = [n for n, _ in type(v0)._fields_ if as_list(getattr(v0, n)) != as_list(getattr(fast, n))]
    assert sorted(diff) == ["ego_collisions_only", "ego_spacing"]


def test_absent_key_is_highway_v0(highway_config):
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg, resolve_config

    for cfg in (highway_config, {}, {"vehicles_count": 10}):
        named = dict(copy.deepcopy(cfg), gym_id="highway-v0")
        a, b = build_cfg(cfg), build_cfg(named)
        assert bytes(a) == bytes(b) and a.ego_collisions_only == 0
        assert resolve_config(cfg)["gym_id"] == "highway-v0"


def test_unknown_id_is_a_value_error_before_any_device_work(highway_config):
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_env

    with pytest.raises(ValueError, match="highway-fast-v0"):
        build_cfg({"gym_id": "merge-v0"})
    with pytest.raises(ValueError, match="'highway-v0', 'highway-fast-v0'"):
        make_env(Condition.SORTED, dict(highway_config, gym_id="highway-v1"))


def test_translation_matches_the_oracle_on_fast_configs(highway_config):
    """the comparison of tests/test_abi_cpu.py test_config_translation_matches_oracle_translation on fast configs"""
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    cfgs = [{"gym_id": FAST, "observation": dict(KINEMATICS)}, dict(copy.deepcopy(highway_config), gym_id=FAST),
            {"gym_id": FAST, "vehicles_count": 10, "action": {"type": "ContinuousAction"}}]
    for c in cfgs:
        a, b = build_cfg(c), fast_oh.cfg_from_dict(c)
        for name, _ in oh.HwCfg._fields_:
            if name == "_pad":
                continue
            va, vb = getattr(a, name), getattr(b, name)
            if hasattr(va, "__len__"):
                assert list(va) == list(vb), name
            else:
                assert va == vb, name
        assert a.ego_collisions_only == 1
    assert fast_oh.cfg_from_dict({"gym_id": FAST}).ego_spacing == 1.5 and oh.cfg_from_dict({}).ego_spacing == 2.0


def test_c_abi_field(highway_config):
    from highway_rope_ppo_b200 import _lib
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    lib = _lib.load()
    assert lib.hrp_version() == 3
    for bad in (2, -1):
        c = build_cfg(highway_config)
        c.ego_collisions_only = bad
        h = C.c_void_p()
        assert lib.hrp_env_create_ex(C.byref(c), None, 0, 1, 0, 0, 0, C.byref(h)) == -1
        assert "ego_collisions_only" in _lib.last_error()
    c = build_cfg(dict(highway_config, gym_id=FAST))
    h = C.c_void_p()
    rc = lib.hrp_env_create_ex(C.byref(c), None, 0, 1, 0, 0, 0, C.byref(h))
    if rc == 0:
        lib.hrp_env_destroy(h)
    assert rc == (0 if _lib.device_count() > 0 else -3), _lib.last_error()


# ---- the oracle's collision rule, worked out by hand -----------------------------------------------------------------
# Three vehicles (ego = 0) on 3 lanes at 5 Hz, heading 0, all at 25 m/s, IDM timers at 0 and no lane change under way:
# in the first frame nothing steers, every x advances by the same 5 m, and rectangles of 5 x 2 m that overlap in x on
# one lane intersect (and will intersect).  Frame 0 of the trace holds the flags and the impacts its collisions set.
def _hand_cfg(gym_id):
    return {"gym_id": gym_id, "vehicles_count": 2, "lanes_count": 3, "simulation_frequency": 5,
            "action": {"type": "ContinuousAction"}, "observation": dict(KINEMATICS)}


def _hand_state(placed):
    """placed: [(x, lane)] of the ego and the two other vehicles"""
    V = len(placed)
    st = {k: np.zeros(V) for k in oh.STATE_F64}
    st.update({k: np.zeros(V, dtype=np.int32) for k in oh.STATE_I32})
    st["x"][:] = [p[0] for p in placed]
    st["lane"][:] = st["target_lane"][:] = [p[1] for p in placed]
    st["y"][:] = 4.0 * st["lane"]
    st["speed"][:] = st["target_speed"][:] = 25.0
    st["delta"][:] = 4.0
    st["time"], st["steps"] = 0.0, 0
    return st


HAND_CASES = {   # the states of cases (a) to (d); tests/test_fast_env_gpu.py injects the same ones
    "a": [(0.0, 0), (300.0, 2), (302.0, 2)],      # two uncontrolled vehicles overlapping, far from the ego
    "b": [(100.0, 1), (103.0, 1), (400.0, 2)],    # ego contact
    "c": [(100.0, 1), (97.0, 1), (103.5, 1)],     # the ego overlaps vehicle 1 (behind) and vehicle 2 (ahead)
    "d": [(100.0, 1), (103.5, 1), (107.0, 1)],    # vehicle 1 overlaps the ego (behind it) and vehicle 2 (ahead of it)
}


def _frame0(gym_id, case):
    cfg = _hand_cfg(gym_id)
    o = oracle_module(cfg).OracleEnv(cfg)
    o.set_state(_hand_state(HAND_CASES[case]))
    tr = o.trace()
    o.step(np.zeros(2, np.float32))
    f = tr[0].copy()
    flags = f[:, 6].astype(np.int64)
    return {"x": f[:, 0], "y": f[:, 1], "impact_x": f[:, 4], "impact_y": f[:, 5], "crashed": (flags >> 16) & 1,
            "has_impact": (flags >> 17) & 1}, o.get_state()


def test_a_uncontrolled_pair_collides_only_under_highway_v0():
    v0, _ = _frame0("highway-v0", "a")
    assert list(v0["crashed"]) == [0, 1, 1] and list(v0["has_impact"]) == [0, 1, 1]
    # full overlap across (2 m) beats 3 m along: the impact separates them sideways, 1 m each
    assert v0["impact_y"][1] == pytest.approx(-1.0) and v0["impact_y"][2] == pytest.approx(1.0)
    fast, end = _frame0(FAST, "a")
    assert not fast["crashed"].any() and not fast["has_impact"].any()
    assert not end["crashed"].any() and not end["has_impact"].any()
    assert (end["y"][1:] == 8.0).all() and (end["heading"][1:] == 0.0).all()   # neither displaced


@pytest.mark.parametrize("gym_id", ["highway-v0", FAST])
def test_b_ego_contact_crashes_under_both(gym_id):
    f, end = _frame0(gym_id, "b")
    assert list(f["crashed"]) == [1, 1, 0] and list(f["has_impact"]) == [1, 1, 0]
    assert end["crashed"][0] == 1


@pytest.mark.parametrize("gym_id", ["highway-v0", FAST])
def test_c_the_ego_keeps_the_impact_of_its_last_pair(gym_id):
    f, _ = _frame0(gym_id, "c")
    assert list(f["crashed"]) == [1, 1, 1] and list(f["has_impact"]) == [1, 1, 1]
    # pair (0, 1) would push the ego forward, pair (0, 2) pushes it back by half the 1.5 m overlap (less the closing
    # speed of vehicle 2, which accelerates on a free road while the ego holds 25 m/s)
    assert -0.75 - 1e-2 < f["impact_x"][0] < -0.7 and f["impact_y"][0] == pytest.approx(0.0, abs=1e-12)
    assert f["impact_x"][1] < 0.0 < f["impact_x"][2]   # vehicle 1 pushed back, vehicle 2 forward


def test_d_impact_of_a_vehicle_between_two_pairs():
    v0, _ = _frame0("highway-v0", "d")
    fast, _ = _frame0(FAST, "d")
    # highway-v0: pair (1, 2) comes after (0, 1) and pushes vehicle 1 back; highway-fast-v0 tests (0, 1) only, which
    # pushes it forward
    assert v0["impact_x"][1] < -0.5 and fast["impact_x"][1] > 0.5
    assert list(v0["crashed"]) == [1, 1, 1] and list(fast["crashed"]) == [1, 1, 0]
    assert v0["has_impact"][2] == 1 and fast["has_impact"][2] == 0
    assert v0["impact_x"][0] == fast["impact_x"][0] < 0.0


def test_main_gym_id_flag(capsys):
    from highway_rope_ppo_b200 import main

    assert main.parse([]).gym_id is None
    assert main.parse(["--gym-id", FAST]).gym_id == FAST
    with pytest.raises(SystemExit):
        main.parse(["--gym-id", "merge-v0"])
    capsys.readouterr()
    assert main.main(["--get-total-experiments"]) == 0
    plain = capsys.readouterr().out
    assert main.main(["--get-total-experiments", "--gym-id", FAST]) == 0
    assert capsys.readouterr().out == plain and int(plain) > 0


def test_main_puts_the_key_into_the_base_config(monkeypatch):
    from highway_rope_ppo_b200 import main
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.experiments import sweep
    from highway_rope_ppo_b200.utils.reproducibility import SEED

    name = sweep.define_experiments(SEED, 3)[0].name
    seen = []
    monkeypatch.setattr(sweep, "run_experiments", lambda mine, base, **kw: seen.append(base) or [])
    for argv, want in (([], None), (["--gym-id", FAST], FAST)):
        main.main(argv + ["--run-single-experiment", name, "--max-episodes", "1"])
        base = seen.pop()
        assert base.get("gym_id") == want
        assert {k: v for k, v in base.items() if k != "gym_id"} == HIGHWAY_CONFIG
    assert "gym_id" not in HIGHWAY_CONFIG
