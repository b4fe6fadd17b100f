"""ctypes binding of ``libhrp_b200.so`` (``include/hrp.h``).

The library is the product: there is no Python or CPU fallback behind these calls.  If the
shared object is missing the import of any compute module fails with instructions to build it;
if no CUDA device is present every compute entry point raises ``HrpError``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Any, Dict, Optional

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "lib", "libhrp_b200.so")

HRP_MAX_VEHICLES = 64
HRP_MAX_OBS_ROWS = 64
HRP_MAX_FEATURES = 8
HRP_MAX_LANES = 8
HRP_MAX_EMBED = 64

HRP_MAX_GRID_VALUES = HRP_MAX_OBS_ROWS * HRP_MAX_FEATURES   # F * W * H of an OccupancyGrid observation

# "on_road" (HRP_F_ON_ROAD) is the OccupancyGrid road layer: valid in a grid only
FEATURE_CODES = {"presence": 0, "x": 1, "y": 2, "vx": 3, "vy": 4, "heading": 5, "cos_h": 6, "sin_h": 7, "on_road": 8}
OBS_KINEMATICS, OBS_OCCUPANCY_GRID = 0, 1   # HRP_OBS_*
EMBED_NONE, EMBED_ROPE, EMBED_DIST, EMBED_RANK = 0, 1, 2, 3
PPO_CATEGORICAL = 1   # HRP_PPO_CATEGORICAL
EPISODE_STATS_LEN = 6 + 6 * 512   # HRP_EPISODE_STATS_LEN: doubles of hrp_episode_stats' stats_dev
VECNORM_MAX_S = 4608                # HRP_VECNORM_MAX_S: 64 rows x (8 features + 64 embedding columns)
VECNORM_MAX_E = 1 << 24             # HRP_VECNORM_MAX_E


def vecnorm_moments_len(C: int) -> int:
    """HRP_VECNORM_MOMENTS_LEN: doubles of one rank's batch moments over C columns."""
    return 1 + 2 * C


def vecnorm_scratch_len(C: int) -> int:
    """HRP_VECNORM_SCRATCH_LEN: doubles of the scratch of hrp_vecnorm_moments / hrp_vecnorm_merge."""
    return 256 + 256 * C


class HrpError(RuntimeError):
    """A call into libhrp_b200.so failed (message from hrp_last_error())."""


class HrpCfg(C.Structure):
    _fields_ = [
        ("lanes_count", C.c_int32), ("vehicles_count", C.c_int32),
        ("simulation_frequency", C.c_int32), ("policy_frequency", C.c_int32),
        ("initial_lane_id", C.c_int32), ("ego_mode", C.c_int32),
        ("normalize_reward", C.c_int32), ("offroad_terminal", C.c_int32),
        ("duration", C.c_double), ("ego_spacing", C.c_double), ("vehicles_density", C.c_double),
        ("collision_reward", C.c_double), ("right_lane_reward", C.c_double),
        ("high_speed_reward", C.c_double), ("reward_speed_lo", C.c_double),
        ("reward_speed_hi", C.c_double),
        ("obs_vehicles", C.c_int32), ("obs_nfeat", C.c_int32),
        ("obs_feat", C.c_int32 * HRP_MAX_FEATURES), ("obs_has_range", C.c_int32 * HRP_MAX_FEATURES),
        ("obs_lo", C.c_double * HRP_MAX_FEATURES), ("obs_hi", C.c_double * HRP_MAX_FEATURES),
        ("obs_normalize", C.c_int32), ("obs_clip", C.c_int32), ("obs_absolute", C.c_int32),
        ("obs_sorted", C.c_int32), ("obs_see_behind", C.c_int32),
        ("embed_kind", C.c_int32), ("embed_dim", C.c_int32), ("embed_use_euclidean", C.c_int32),
        ("embed_max_dist", C.c_double),
        ("autoreset", C.c_int32), ("embed_ego_idx", C.c_int32),
        ("obs_type", C.c_int32), ("grid_align", C.c_int32),
        ("grid_lo", C.c_double * 2), ("grid_hi", C.c_double * 2), ("grid_step", C.c_double * 2),
        ("ego_collisions_only", C.c_int32),
    ]


class HrpState(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_double)) for n in
                ("x", "y", "heading", "speed", "target_speed", "delta", "timer", "impact_x", "impact_y")] + \
               [(n, C.POINTER(C.c_int32)) for n in ("lane", "target_lane", "crashed", "has_impact")] + \
               [("time", C.POINTER(C.c_double)), ("episode", C.POINTER(C.c_uint32)),
                ("obs_draw", C.POINTER(C.c_uint32))]


class HrpActItem(C.Structure):
    """``hrp_act_item``: one policy / one state of ``hrp_ppo_act_multi``."""
    _fields_ = [("params_dev", C.c_void_p), ("state_dev", C.c_void_p), ("out_dev", C.c_void_p),
                ("seed", C.c_uint64), ("draw", C.c_uint64), ("row", C.c_uint64),
                ("state_dim", C.c_int32), ("action_dim", C.c_int32), ("hidden_dim", C.c_int32),
                ("deterministic", C.c_int32)]


STATE_F64 = ("x", "y", "heading", "speed", "target_speed", "delta", "timer", "impact_x", "impact_y")
STATE_I32 = ("lane", "target_lane", "crashed", "has_impact")

_vp, _i32, _i64, _u64, _f32, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_double

# name -> (restype, argtypes): every symbol include/hrp.h declares
SIGNATURES: Dict[str, Any] = {
    "hrp_last_error": (C.c_char_p, []),
    "hrp_version": (C.c_int, []),
    "hrp_device_count": (C.c_int, []),
    "hrp_env_create": (C.c_int, [C.POINTER(HrpCfg), _vp, _i64, _i32, _u64, _i32, C.POINTER(_vp)]),
    "hrp_env_create_ex": (C.c_int, [C.POINTER(HrpCfg), _vp, _i64, _i32, _u64, _i32, C.c_uint32, C.POINTER(_vp)]),
    "hrp_env_destroy": (C.c_int, [_vp]),
    "hrp_env_obs_dim": (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_i32)]),
    "hrp_env_grid_shape": (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "hrp_env_num_vehicles": (C.c_int, [_vp]),
    "hrp_env_reset": (C.c_int, [_vp, _u64, _vp, _vp, _vp]),
    "hrp_env_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hrp_env_step_final": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hrp_env_observe": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "hrp_env_step_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "hrp_env_reset_host": (C.c_int, [_vp, _u64, _vp]),
    "hrp_env_step_host_on": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hrp_fetch_host": (C.c_int, [_vp, _vp, _u64, _vp]),
    "hrp_env_set_seeds": (C.c_int, [_vp, _vp]),
    "hrp_env_set_step_mask": (C.c_int, [_vp, _vp]),
    "hrp_env_set_trace": (C.c_int, [_vp, _vp]),
    "hrp_env_trace_shape": (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "hrp_env_step_host_async": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hrp_env_get_state": (C.c_int, [_vp, C.POINTER(HrpState)]),
    "hrp_env_set_state": (C.c_int, [_vp, C.POINTER(HrpState)]),
    "hrp_philox4x32_10": (C.c_int, [_vp, _vp, _vp]),
    "hrp_embed_apply": (C.c_int, [_i32, _i32, _i32, _i32, _f32, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp]),
    "hrp_ppo_param_count": (_i64, [_i32, _i32, _i32]),
    "hrp_ppo_param_count_ex": (_i64, [_i32, _i32, _i32, C.c_uint32]),
    "hrp_ppo_set_math": (C.c_int, [_i32]),
    "hrp_ppo_get_math": (C.c_int, []),
    "hrp_gemm_strided": (C.c_int, [_i32, _i32, _i32, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i32, _vp, _i32, _i32, _vp]),
    "hrp_ppo_create": (C.c_int, [_i32, _i32, _i32, _i64, _i32, C.POINTER(_vp)]),
    "hrp_ppo_create_ex": (C.c_int, [_i32, _i32, _i32, _i64, _i32, C.c_uint32, C.POINTER(_vp)]),
    "hrp_ppo_destroy": (C.c_int, [_vp]),
    "hrp_ppo_forward": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "hrp_ppo_act": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hrp_ppo_act_sample": (C.c_int, [_vp, _vp, _vp, _u64, _u64, _u64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hrp_ppo_act_multi": (C.c_int, [_vp, _i32, _vp]),
    "hrp_ppo_act_sample_ctr": (C.c_int, [_vp, _vp, _vp, _u64, _vp, _u64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hrp_gae": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _f64, _f64, _vp, _vp, _vp]),
    "hrp_gae_ex": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _f64, _f64, _vp, _vp, _vp]),
    "hrp_adv_stats": (C.c_int, [_vp, _i64, _vp, _vp]),
    "hrp_adv_normalize": (C.c_int, [_vp, _i64, _vp, _vp]),
    "hrp_episode_stats": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hrp_ppo_loss_grad": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp,
                                    _vp, _vp]),
    "hrp_ppo_loss_grad_ex": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp,
                                       _f32, _vp, _vp, _vp]),
    "hrp_clip_adam_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _f64, _f64, _f64, _f64, _f32, _vp, _vp]),
    "hrp_clip_adam_step_ex": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _f64, _vp, _f64, _f64, _f64, _f32, _vp, _vp]),
    "hrp_ppo_loss_grad_kl": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _vp,
                                       _f32, _vp, _vp, _vp, _vp, _vp]),
    "hrp_clip_adam_step_kl": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _f64, _vp, _f64, _f64, _f64, _f32, _vp, _vp, _vp,
                                        _f64, _vp]),
    "hrp_graph_if_create": (C.c_int, [_vp, _vp, _vp, C.POINTER(_vp)]),
    "hrp_graph_if_launch": (C.c_int, [_vp, _vp]),
    "hrp_graph_if_destroy": (C.c_int, [_vp]),
    "hrp_comm_create": (C.c_int, [_i32, _i32, _i64, _i32, C.POINTER(_vp), _vp]),
    "hrp_comm_connect": (C.c_int, [_vp, _vp]),
    "hrp_comm_grad": (_vp, [_vp]),
    "hrp_comm_grad_parity": (_vp, [_vp, _i32]),
    "hrp_comm_parity": (C.c_int, [_vp]),
    "hrp_comm_note_replay": (C.c_int, [_vp]),
    "hrp_clip_adam_step_p2p": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _f64, _f64, _f64, _f64, _f32, _vp, _vp]),
    "hrp_clip_adam_step_p2p_ex": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _f64, _vp, _f64, _f64, _f64, _f32, _vp, _vp]),
    "hrp_clip_adam_step_p2p_kl": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _f64, _vp, _f64, _f64, _f64, _f32, _vp, _vp, _f64,
                                            _vp]),
    "hrp_vecnorm_moments": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _f64, _vp, _vp, _vp]),
    "hrp_vecnorm_merge": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "hrp_vecnorm_apply": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _f64, _f64, _f64, _vp]),
    "hrp_comm_status": (C.c_int, [_vp]),
    "hrp_comm_destroy": (C.c_int, [_vp]),
}

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the shared object and type every entry point.  Raises ImportError when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python highway-rope-ppo_b200/build.py` "
            "(or __graft_entry__.build()); the framework has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().hrp_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise HrpError(f"{what or 'libhrp_b200'} failed (rc={rc}): {last_error()}")


def device_count() -> int:
    return int(load().hrp_device_count())


def require_device() -> None:
    n = device_count()
    if n <= 0:
        raise HrpError("no CUDA device visible: highway-rope-ppo_b200 has no CPU path "
                       f"(hrp_device_count() = {n}: {last_error()})")


def ptr(t) -> Optional[int]:
    """data pointer of a torch tensor / numpy array (None passes NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def stream_ptr(device) -> int:
    import torch

    return torch.cuda.current_stream(device).cuda_stream
