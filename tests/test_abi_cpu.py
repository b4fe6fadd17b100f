"""CPU-side checks of the boundary: the library loads, exports every symbol include/hrp.h declares, the
ctypes mirror of hrp_cfg has the C layout, config translation and the reference's error behaviour hold,
and compute entry points fail loudly (no CPU fallback) when no device is visible."""
import copy
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "hrp.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hrp_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), name
    assert sorted(_lib.SIGNATURES) == declared
    assert lib.hrp_version() >= 1


def test_cfg_struct_layout_matches_c(tmp_path):
    """sizeof/offsetof of hrp_cfg as gcc sees include/hrp.h == the ctypes mirror."""
    from highway_rope_ppo_b200._lib import HrpCfg, HrpState

    src = tmp_path / "l.c"
    fields = [f[0] for f in HrpCfg._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hrp.h"\nint main(){printf("%zu %zu", sizeof(hrp_cfg), sizeof(hrp_state));'
                   + "".join(f'printf(" %zu", offsetof(hrp_cfg, {f}));' for f in fields) + "return 0;}\n")
    exe = tmp_path / "l"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    nums = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert nums[0] == C.sizeof(HrpCfg) and nums[1] == C.sizeof(HrpState)
    assert nums[2:] == [getattr(HrpCfg, f).offset for f in fields]


def test_act_item_struct_layout_matches_c(tmp_path):
    """hrp_act_item (hrp_ppo_act_multi) as gcc sees it == the ctypes mirror."""
    from highway_rope_ppo_b200._lib import HrpActItem

    src = tmp_path / "a.c"
    fields = [f[0] for f in HrpActItem._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hrp.h"\nint main(){printf("%zu", sizeof(hrp_act_item));'
                   + "".join(f'printf(" %zu", offsetof(hrp_act_item, {f}));' for f in fields) + "return 0;}\n")
    exe = tmp_path / "a"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    nums = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert nums[0] == C.sizeof(HrpActItem) == 64
    assert nums[1:] == [getattr(HrpActItem, f).offset for f in fields]


def test_philox_host_entry_point_known_answer():
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    ctr = np.array([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], dtype=np.uint32)
    key = np.array([0xa4093822, 0x299f31d0], dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    assert lib.hrp_philox4x32_10(ctr.ctypes.data, key.ctypes.data, out.ctypes.data) == 0
    assert [hex(int(x)) for x in out] == ["0xd16cfe09", "0x94fdcceb", "0x5001e420", "0x24126ea1"]


def test_param_count_matches_reference_architecture():
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    assert lib.hrp_ppo_param_count(60, 2, 256) == 213765   # SURVEY 8c
    assert lib.hrp_ppo_param_count(60, 2, 512) == 820741   # SURVEY 8d config 4
    assert lib.hrp_ppo_param_count(600, 2, 512) == 1097221


def test_config_translation_matches_oracle_translation(highway_config):
    """The product's dict -> hrp_cfg and the oracle's dict -> hw_cfg agree on every shared field."""
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg
    from oracle import highway as oh

    cfg = copy.deepcopy(highway_config)
    cfg["observation"]["features"] = ["presence", "x", "y", "vx", "vy", "cos_h", "sin_h"]
    for c in (highway_config, cfg, {"vehicles_count": 10}):
        a, b = build_cfg(c), oh.cfg_from_dict(c)
        for name, _ in oh.HwCfg._fields_:
            if name == "_pad":
                continue
            va, vb = getattr(a, name), getattr(b, name)
            if hasattr(va, "__len__"):
                assert list(va) == list(vb), name
            else:
                assert va == vb, name
    assert build_cfg(highway_config).ego_mode == 0 and build_cfg(highway_config).vehicles_density == 2.0


def test_config_errors():
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    with pytest.raises(ValueError):
        build_cfg({"observation": {"type": "GrayscaleObservation"}})
    with pytest.raises(ValueError):
        build_cfg({"observation": {"type": "Kinematics", "features": ["x", "bogus"]}})
    with pytest.raises(ValueError):
        build_cfg({"action": {"type": "ContinuousAction", "lateral": False}})
    with pytest.raises(ValueError):
        build_cfg({"observation": {"type": "Kinematics", "order": "random"}})


def test_make_env_validation_happens_before_any_device_work(highway_config):
    """The reference's early ValueErrors (wrappers.py:61-71) need no GPU."""
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import _resolve, make_env

    with pytest.raises(ValueError, match="rotate_dim"):
        make_env(Condition.SHUFFLED_ROPE, highway_config, d_embed=16)
    with pytest.raises(ValueError, match="DistPE"):
        make_env(Condition.SHUFFLED_DISTPE, highway_config, d_embed=5)
    # setdefault semantics (SURVEY F3) and deep-merge of overrides, without mutating the base config
    before = copy.deepcopy(highway_config)
    assert _resolve(Condition.SHUFFLED, highway_config, None, {})["observation"]["order"] == "sorted"
    merged = _resolve(Condition.SHUFFLED, highway_config, None, {"observation": {"order": "shuffled"}, "duration": 7})
    assert merged["observation"]["order"] == "shuffled" and merged["observation"]["vehicles_count"] == 15
    assert merged["duration"] == 7 and highway_config == before


def test_defaults_match_config(highway_config):
    """The reference's tests/test_defaults.py:4-17."""
    from highway_rope_ppo_b200.utils.defaults import feature_count, max_dist, max_rank

    r = highway_config["observation"]["features_range"]
    assert max_dist() == max(abs(r["x"][0]), abs(r["x"][1]), abs(r["y"][0]), abs(r["y"][1])) == 100
    assert max_rank() == highway_config["observation"]["vehicles_count"] == 15
    assert feature_count() == len(highway_config["observation"]["features"]) == 4


def test_sweep_expansion():
    from highway_rope_ppo_b200.experiments.config import ConditionHP, expand_condition_hps

    hp = ConditionHP(sweep={"lr": [1e-4, 3e-4], "hidden_dim": [256, 384, 512]})
    out = expand_condition_hps(hp)
    assert len(out) == 6 and all(not h.sweep for h in out)
    assert {(h.lr, h.hidden_dim) for h in out} == {(a, b) for a in (1e-4, 3e-4) for b in (256, 384, 512)}


_F8 = ["presence", "x", "y", "vx", "vy", "heading", "cos_h", "sin_h"]
# (case, config overrides, embedding (kind, d, use_euclidean, ego_idx) or None, accepted, what the error names)
_CFG_EDGES = [
    ("vehicles 63", dict(vehicles_count=63), None, True, None),
    ("vehicles 64", dict(vehicles_count=64), None, False, "vehicles_count"),
    ("lanes 1", dict(lanes_count=1), None, True, None),
    ("lanes 0", dict(lanes_count=0), None, False, "lanes_count"),
    ("lanes 8", dict(lanes_count=8), None, True, None),
    ("lanes 9", dict(lanes_count=9), None, False, "lanes_count"),
    ("rows 64", dict(observation=dict(vehicles_count=64)), None, True, None),
    ("rows 65", dict(observation=dict(vehicles_count=65)), None, False, "observation vehicles_count"),
    ("features 8", dict(observation=dict(features=_F8)), None, True, None),
    ("features 9", dict(observation=dict(features=_F8)), None, False, "feature count"),   # obs_nfeat forced to 9
    ("sim = policy", dict(simulation_frequency=3, policy_frequency=3), None, True, None),
    ("sim < policy", dict(simulation_frequency=2, policy_frequency=3), None, False, "frequency"),
    ("rope d = F", {}, ("rope", 4, True, 0), True, None),
    ("rope d = F + 2", {}, ("rope", 6, True, 0), False, "rotate_dim"),
    ("rope d odd", {}, ("rope", 3, True, 0), False, "rotate_dim"),
    ("rope F = 1", dict(observation=dict(features=["presence"])), ("rope", 0, True, 0), False, "RoPE needs"),
    ("dist d 64", {}, ("dist", 64, True, 0), True, None),
    ("dist d 66", {}, ("dist", 66, True, 0), False, "DistPE d_embed"),
    ("dist d odd", {}, ("dist", 7, True, 0), False, "DistPE d_embed"),
    ("dist F = 1 |dx|", dict(observation=dict(features=["x"])), ("dist", 4, False, 0), True, None),
    ("dist F = 1 euclid", dict(observation=dict(features=["x"])), ("dist", 4, True, 0), False, "DistPE needs"),
    ("rank d 1", {}, ("rank", 1, True, 0), True, None),
    ("rank d 64", {}, ("rank", 64, True, 0), True, None),
    ("rank d 65", {}, ("rank", 65, True, 0), False, "RankPE d_embed"),
    ("ego_idx N-1", {}, ("rope", 4, True, 14), True, None),
    ("ego_idx N", {}, ("rope", 4, True, 15), False, "ego_idx"),
]


@pytest.mark.parametrize("case,over,emb,accepted,field", _CFG_EDGES, ids=[c[0] for c in _CFG_EDGES])
def test_env_config_limits(highway_config, case, over, emb, accepted, field):
    """Both sides of every limit hrp_env_create_ex checks.  The configuration is validated before the device is looked
    at: without a GPU an accepted configuration gets -3 (no CUDA device), a rejected one -1 and a message naming the
    field; with a GPU an accepted configuration creates a handle."""
    from highway_rope_ppo_b200 import _lib
    from highway_rope_ppo_b200.envs.highway_vec import EmbedSpec, build_cfg

    lib = _lib.load()
    cfg = copy.deepcopy(highway_config)
    for k, v in over.items():
        if isinstance(v, dict):
            cfg[k].update(v)
        else:
            cfg[k] = v
    spec = None
    if emb is not None:
        kind, d, eu, ego = emb
        kind = {"rope": _lib.EMBED_ROPE, "dist": _lib.EMBED_DIST, "rank": _lib.EMBED_RANK}[kind]
        spec = EmbedSpec(kind, d, use_euclidean=eu, ego_idx=ego)
    c = build_cfg(cfg, spec)
    if case == "features 9":
        with pytest.raises(ValueError):
            build_cfg(dict(cfg, observation=dict(cfg["observation"], features=_F8 + ["x"])))
        c.obs_nfeat = 9
    n = 0
    if emb is not None:   # the table length each kind expects, so that only the field under test can be wrong
        n = c.obs_vehicles * d if emb[0] == "rank" else d // 2
    table = np.zeros(max(n, 1), dtype=np.float32)
    h = C.c_void_p()
    rc = lib.hrp_env_create_ex(C.byref(c), table.ctypes.data if emb is not None else None, n, 4, 0, 0, 0, C.byref(h))
    if accepted:
        has_device = lib.hrp_device_count() > 0
        assert rc == (0 if has_device else -3), (rc, _lib.last_error())
        if rc == 0:
            assert lib.hrp_env_destroy(h) == 0
    else:
        assert rc == -1 and field in _lib.last_error(), (rc, _lib.last_error())


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device behaviour")
def test_no_cpu_fallback(highway_config):
    from highway_rope_ppo_b200 import _lib
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    with pytest.raises(_lib.HrpError):
        HighwayVecEnv(highway_config, 4)
    with pytest.raises(_lib.HrpError):
        PPOAgent(60, 2, device="cpu")
    with pytest.raises(_lib.HrpError):
        PPOAgent(60, 2, device="cuda:0")


def test_wrapper_constructor_errors_without_device():
    from highway_rope_ppo_b200.envs.spaces import Box
    from highway_rope_ppo_b200.experiments.dist_embed import DistanceEmbedWrapper
    from highway_rope_ppo_b200.experiments.rank_embed import RankEmbedWrapper
    from highway_rope_ppo_b200.experiments.rope_embed import RotaryEmbedWrapper

    class E:
        def __init__(self, shape):
            self.observation_space = Box(-np.inf, np.inf, shape, np.float32)
            self.action_space = Box(-1, 1, (2,), np.float32)

    with pytest.raises(ValueError):
        RotaryEmbedWrapper(E((5, 4)), rotate_dim=3)
    with pytest.raises(ValueError):
        RotaryEmbedWrapper(E((5, 4)), rotate_dim=6)
    assert RotaryEmbedWrapper(E((4, 4)), max_dist=1.0).rotate_dim == 4
    assert RotaryEmbedWrapper(E((4, 5)), max_dist=1.0).rotate_dim == 4
    np.testing.assert_allclose(RotaryEmbedWrapper(E((15, 4)), rotate_dim=4).inv_freq, [1.0, 0.1], rtol=1e-6)
    with pytest.raises(ValueError):
        DistanceEmbedWrapper(E((5, 4)), d_embed=3)
    with pytest.raises(ValueError):
        DistanceEmbedWrapper(E((5, 1)), d_embed=4)
    with pytest.raises(ValueError):
        DistanceEmbedWrapper(E((5,)), d_embed=4)
    with pytest.raises(ValueError):
        RankEmbedWrapper(E((5,)), d_embed=4)
    with pytest.raises(TypeError):
        class NotBox:
            observation_space = object()
        RankEmbedWrapper(NotBox(), d_embed=4)
    w = DistanceEmbedWrapper(E((15, 4)), d_embed=16)
    assert w.observation_space.shape == (15, 20)
    torch.manual_seed(42)
    r = RankEmbedWrapper(E((15, 4)), d_embed=4)
    assert r.observation_space.shape == (15, 8) and float(r.table.weight.abs().max()) <= 0.05
