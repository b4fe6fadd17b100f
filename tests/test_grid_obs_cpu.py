"""OccupancyGrid observation, CPU side: the fp64 restatement against grids worked out by hand, and the config / C ABI
errors, which are raised before any device work."""
import ctypes as C
import math

import numpy as np
import pytest

from grid_oracle import GridOracle

EGO_X, EGO_Y = 500.0, 4.0   # lane 1 of 4, far from both road ends


def _state(*vehicles):
    """vehicles as (dx, dy, heading, speed) relative to the ego at (EGO_X, EGO_Y) with heading 0, speed 0"""
    rows = [(0.0, 0.0, 0.0, 0.0)] + list(vehicles)
    x = [EGO_X + r[0] for r in rows]
    y = [EGO_Y + r[1] for r in rows]
    return x, y, [r[2] for r in rows], [r[3] for r in rows]


def test_ego_owns_the_centre_cell_with_zero_velocity():
    o = GridOracle()
    grid, cells = o.observe(*_state())
    assert grid.shape == (4, 11, 11) and o.shape == (4, 11, 11)
    assert cells.reshape(11, 11)[5, 5] == 0 and (cells >= 0).sum() == 1
    assert grid[0, 5, 5] == 1.0 and grid[0].sum() == 1.0
    assert grid[1, 5, 5] == 0.0 and grid[2, 5, 5] == 0.0


def test_vehicle_at_dx12_dy4_lands_in_cell_7_6():
    o = GridOracle()
    grid, cells = o.observe(*_state((12.0, 4.0, 0.0, 8.0)))
    assert cells.reshape(11, 11)[7, 6] == 1
    assert grid[0, 7, 6] == 1.0
    assert grid[1, 7, 6] == np.float32(-1 + (8.0 + 80.0) * 2 / 160.0)   # vx relative to a resting ego, lmap'd
    assert grid[2, 7, 6] == 0.0


def test_lower_index_wins_a_shared_cell():
    o = GridOracle(features=["presence", "vx"])
    grid, cells = o.observe(*_state((12.0, 4.0, 0.0, 8.0), (10.0, 4.5, 0.0, 40.0)))
    assert cells.reshape(11, 11)[7, 6] == 1
    assert grid[1, 7, 6] == np.float32(-1 + 88.0 * 2 / 160.0)
    # in the other list order the other vehicle wins
    grid, cells = o.observe(*_state((10.0, 4.5, 0.0, 40.0), (12.0, 4.0, 0.0, 8.0)))
    assert cells.reshape(11, 11)[7, 6] == 1 and grid[1, 7, 6] == np.float32(-1 + 120.0 * 2 / 160.0)


def test_left_edge_is_column_0_and_right_edge_is_dropped():
    o = GridOracle(features=["presence"])
    grid, cells = o.observe(*_state((-27.5, 0.0, 0.0, 0.0), (27.5, 0.0, 0.0, 0.0)))
    c = cells.reshape(11, 11)
    assert c[0, 5] == 1
    assert 2 not in cells
    assert grid[0].sum() == 2.0


def test_on_road_rows_for_ego_on_lane_1_of_4():
    o = GridOracle(features=["on_road"], lanes=4)
    grid, _ = o.observe(*_state())
    want = np.zeros((11, 11), np.float32)
    want[:, 4:8] = 1.0   # lanes 0..3 at y - 4 = -4, 0, 4, 8: rows floor((dy + 27.5) / 5) = 4, 5, 6, 7
    assert np.array_equal(grid[0], want)


def test_on_road_is_clipped_to_the_road_near_its_start():
    o = GridOracle(features=["on_road"], lanes=1)
    x, y, h, v = _state()
    grid, _ = o.observe([10.0], [0.0], h, v)   # ego at x = 10: waypoints below 0 collapse onto x = 0 (column 3)
    assert grid[0, :, 5].tolist() == [0.0] * 3 + [1.0] * 8


def test_rotated_grid():
    o = GridOracle(features=["presence"], align_to_vehicle_axes=True)
    x, y, h, v = _state((0.0, 12.0, 0.0, 0.0))
    h[0] = math.pi / 2   # the ego faces +y: a vehicle 12 m to its +y side is 12 m ahead in its own axes
    grid, cells = o.observe(x, y, h, v)
    c = cells.reshape(11, 11)
    assert c[7, 5] == 1 and c[5, 5] == 0
    # (dx, dy) = (12, 0) is on its right: [[c, s], [-s, c]] @ (12, 0) = (~0, -12)
    x, y, h, v = _state((12.0, 0.0, 0.0, 0.0))
    h[0] = math.pi / 2
    _, cells = o.observe(x, y, h, v)
    assert cells.reshape(11, 11)[5, 3] == 1


def test_xy_features_range_round_trip():
    rng = {"x": [-100.0, 100.0], "y": [-100.0, 100.0]}
    o = GridOracle(features=["presence", "x", "y"], features_range=rng)
    grid, cells = o.observe(*_state((12.0, 4.0, 0.0, 0.0)))
    assert cells.reshape(11, 11)[7, 6] == 1
    assert grid[1, 7, 6] == np.float32(-1 + 112.0 * 2 / 200.0) and grid[2, 7, 6] == np.float32(-1 + 104.0 * 2 / 200.0)
    # a position exactly on a boundary stays there through the round trip: dx = -22.5 -> column 1
    _, cells = o.observe(*_state((-22.5, 0.0, 0.0, 0.0)))
    assert cells.reshape(11, 11)[1, 5] == 1


def test_clip_and_nan_to_zero():
    kw = dict(features=["presence", "vx"], features_range={"vx": [-5.0, 5.0]})
    st = _state((12.0, 4.0, 0.0, 20.0))
    grid, _ = GridOracle(clip=True, **kw).observe(*st)
    assert grid[1, 7, 6] == 1.0                           # lmap(20, [-5, 5], [-1, 1]) = 4, clipped
    assert np.count_nonzero(grid[1]) == 1 and not np.isnan(grid).any()
    grid, _ = GridOracle(clip=False, **kw).observe(*st)
    assert grid[1, 7, 6] == 4.0 and np.count_nonzero(grid[1]) == 1
    # an un-normalised feature is clipped too
    grid, _ = GridOracle(features=["x"], features_range={}, clip=True).observe(*st)
    assert grid[0, 7, 6] == 1.0
    grid, _ = GridOracle(features=["x"], features_range={}, clip=False).observe(*st)
    assert grid[0, 7, 6] == 12.0


def test_marginal_floor_is_keyed_and_forceable():
    o = GridOracle(features=["presence"])
    o.record_below = 1e-3
    st = _state((12.5 - 1e-6, 0.0, 0.0, 0.0))   # a hair left of the boundary between columns 7 and 8
    _, cells = o.observe(*st)
    assert cells.reshape(11, 11)[7, 5] == 1 and ("veh", 1, 0) in o.marginal
    o.forced = {("veh", 1, 0)}
    _, cells = o.observe(*st)
    assert cells.reshape(11, 11)[8, 5] == 1


# ---- config and C ABI errors ------------------------------------------------------------------------------------
GRID = {"type": "OccupancyGrid"}


def _cfg(obs, **env):
    c = {"observation": obs, "action": {"type": "ContinuousAction"}}
    c.update(env)
    return c


def test_resolve_config_applies_grid_defaults():
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg, resolve_config

    obs = resolve_config(_cfg(dict(GRID)))["observation"]
    assert obs["features"] == ["presence", "vx", "vy", "on_road"]
    assert obs["grid_size"] == [[-27.5, 27.5], [-27.5, 27.5]] and obs["grid_step"] == [5, 5]
    assert obs["align_to_vehicle_axes"] is False and obs["clip"] is True
    c = build_cfg(_cfg(dict(GRID)))
    assert c.obs_type == 1 and c.obs_nfeat == 4 and list(c.obs_feat[:4]) == [0, 3, 4, 8]
    assert list(c.obs_has_range[:4]) == [0, 1, 1, 0] and (c.obs_lo[1], c.obs_hi[1]) == (-80.0, 80.0)
    assert list(c.grid_lo) == [-27.5, -27.5] and list(c.grid_hi) == [27.5, 27.5] and list(c.grid_step) == [5.0, 5.0]
    # Kinematics leftovers are ignored; a user features_range replaces the default entirely
    c = build_cfg(_cfg(dict(GRID, vehicles_count=15, order="shuffled", normalize=False, features_range={"vy": [-1, 1]})))
    assert list(c.obs_has_range[:4]) == [0, 0, 1, 0] and c.embed_kind == 0


@pytest.mark.parametrize("bad, what", [
    ({"absolute": True}, "absolute"),
    ({"as_image": True}, "as_image"),
    ({"grid_size": [[-50, 50], [-50, 50]], "grid_step": [2, 2]}, "F x W x H"),
    ({"grid_step": [0, 5]}, "grid_step"),
    ({"grid_size": [[0, 3], [0, 10]]}, "W, H"),
    ({"features": ["presence", "speed"]}, "not implemented"),
])
def test_grid_config_errors(bad, what):
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    with pytest.raises(ValueError, match=what):
        build_cfg(_cfg(dict(GRID, **bad)))


def test_on_road_is_a_grid_feature_only():
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    with pytest.raises(ValueError, match="on_road"):
        build_cfg(_cfg({"type": "Kinematics", "features": ["presence", "on_road"]}))


def test_largest_grid_is_accepted():
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    c = build_cfg(_cfg(dict(GRID, features=["presence", "on_road"], grid_size=[[0, 16], [0, 16]], grid_step=[1, 1])))
    assert c.obs_nfeat * 16 * 16 == 512


@pytest.mark.parametrize("cond", ["SHUFFLED_ROPE", "SHUFFLED_DISTPE", "SHUFFLED_RANKPE"])
def test_embedding_conditions_are_refused_on_a_grid(cond):
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.experiments.config import Condition
    from highway_rope_ppo_b200.experiments.wrappers import make_env, make_vec_env

    over = {"observation": dict(GRID)}
    with pytest.raises(ValueError, match="OccupancyGrid"):
        make_vec_env(Condition[cond], HIGHWAY_CONFIG, d_embed=4, env_overrides=over, num_envs=2)
    with pytest.raises(ValueError, match="OccupancyGrid"):
        make_env(Condition[cond], HIGHWAY_CONFIG, d_embed=4, env_overrides=over)


def _abi_cfg(**kw):
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    c = build_cfg(_cfg(dict(GRID)))
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def _create(c, table=None, n=0):
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.hrp_env_create_ex(C.byref(c), table, n, 1, 0, 0, 0, C.byref(h))
    return rc, _lib.last_error()


def test_c_abi_rejects_bad_grids_before_any_device_query():
    from highway_rope_ppo_b200 import _lib

    assert _lib.load().hrp_version() >= 2
    c = _abi_cfg()
    c.grid_step[0] = 1.0
    c.grid_step[1] = 1.0   # 4 x 55 x 55 values
    rc, msg = _create(c)
    assert rc == -1 and "exceeds 512" in msg
    c = _abi_cfg()
    c.grid_hi[0] = c.grid_lo[0] + 1.0
    rc, msg = _create(c)
    assert rc == -1 and "grid_size[0]" in msg
    c = _abi_cfg()
    c.grid_step[1] = -5.0
    rc, msg = _create(c)
    assert rc == -1 and "grid_step[1]" in msg
    table = (C.c_float * 2)()
    rc, msg = _create(_abi_cfg(embed_kind=1, embed_dim=4), C.cast(table, C.c_void_p), 2)
    assert rc == -1 and "embedding" in msg
    rc, msg = _create(_abi_cfg(obs_type=2))
    assert rc == -1 and "obs_type" in msg


def test_c_abi_rejects_on_road_in_kinematics():
    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    c = build_cfg(_cfg({"type": "Kinematics", "features": ["presence", "x"]}))
    c.obs_feat[1] = 8
    rc, msg = _create(c)
    assert rc == -1 and "feature code 8" in msg


def test_grid_shape_entry_point_is_declared():
    from highway_rope_ppo_b200 import _lib

    assert len(_lib.SIGNATURES["hrp_env_grid_shape"][1]) == 4
    assert _lib.FEATURE_CODES["on_road"] == 8


def test_gpu_parity_configs_fit_the_grid_limit():
    """every grid of tests/test_grid_obs_gpu.py is one the product accepts"""
    from test_grid_obs_gpu import CONFIGS, GRID

    from highway_rope_ppo_b200.envs.highway_vec import build_cfg

    for name, (obs, env) in CONFIGS.items():
        build_cfg(_cfg(dict(GRID, **obs), **env))
