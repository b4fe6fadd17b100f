"""Env factory (reference: ``experiments/wrappers.py:14-104``).

``make_env`` keeps the reference's signature, config handling and error behaviour, and returns a
gymnasium-protocol env whose step runs on the GPU; ``make_vec_env`` is the additive batched
entry point (E lock-step envs, torch tensors in and out) that the vectorised training loop and
``bench.py`` use.
"""
from __future__ import annotations

import copy
from typing import Any, Dict, Optional

from ..envs.highway_env import HighwayEnv
from ..envs.highway_vec import EmbedSpec, HighwayVecEnv, resolve_config
from .config import Condition
from .dist_embed import DistanceEmbedWrapper, dist_freqs
from .rank_embed import RankEmbedWrapper
from .rope_embed import RotaryEmbedWrapper, rope_inv_freq

_SHUFFLED = (Condition.SHUFFLED, Condition.SHUFFLED_RANKPE, Condition.SHUFFLED_DISTPE, Condition.SHUFFLED_ROPE)
_EMBEDDED = (Condition.SHUFFLED_RANKPE, Condition.SHUFFLED_DISTPE, Condition.SHUFFLED_ROPE)


def _merge(dst: Dict[str, Any], src: Dict[str, Any]) -> None:
    """Recursive dict merge: nested dicts are merged, everything else is replaced."""
    for k, v in src.items():
        if isinstance(v, dict) and isinstance(dst.get(k), dict):
            _merge(dst[k], v)
        else:
            dst[k] = v


def _resolve(exp_condition: Condition, base_cfg: Dict[str, Any], d_embed: Optional[int],
             env_overrides: Dict[str, Any]) -> Dict[str, Any]:
    """Steps 1-3 of the reference factory plus its early ``d_embed`` validation."""
    cfg = copy.deepcopy(base_cfg)
    _merge(cfg, env_overrides)
    obs_cfg = cfg.setdefault("observation", {})
    # an OccupancyGrid has no rows to order or to embed: SORTED / SHUFFLED select it unchanged (its `order` is ignored),
    # the embedding conditions are refused before any device work
    if obs_cfg.get("type") == "OccupancyGrid" and exp_condition in _EMBEDDED:
        raise ValueError(f"condition {exp_condition.name} embeds observation rows; an OccupancyGrid observation has none")
    # setdefault: a base config that already names an order keeps it (SURVEY.md F3 -- with the stock
    # HIGHWAY_CONFIG, which says "sorted", the SHUFFLED_* conditions are NOT shuffled unless
    # env_overrides={"observation": {"order": "shuffled"}} is passed)
    if exp_condition is Condition.SORTED:
        obs_cfg.setdefault("order", "sorted")
    elif exp_condition in _SHUFFLED:
        obs_cfg.setdefault("order", "shuffled")
    n_feat = len(cfg["observation"].get("features", []))
    if exp_condition is Condition.SHUFFLED_DISTPE and d_embed is not None:
        if d_embed % 2 != 0 or d_embed > n_feat:
            raise ValueError("d_embed must be even and ≤ feature count for DistPE")
    if exp_condition is Condition.SHUFFLED_ROPE and d_embed is not None:
        if d_embed % 2 != 0 or d_embed > n_feat:
            raise ValueError("rotate_dim (d_embed) must be even and ≤ feature count")
    return cfg


def make_env(exp_condition: Condition, base_cfg: Dict[str, Any], d_embed: Optional[int] = None,
             env_overrides: Dict[str, Any] = {}, device: Any = "cuda"):
    """Create the (wrapped) highway-v0 env for ``exp_condition``.

    Same arguments, config semantics and ``ValueError``s as the reference; ``device`` is additive.
    """
    cfg = _resolve(exp_condition, base_cfg, d_embed, env_overrides)
    env = HighwayEnv(cfg, device=device)
    F = env.observation_space.shape[1]
    if exp_condition is Condition.SHUFFLED_ROPE and d_embed is not None:
        if d_embed % 2 or d_embed > F:
            env.close()
            raise ValueError(f"rotate_dim / d_embed must be even and ≤ {F}")
    if exp_condition is Condition.SHUFFLED_RANKPE:
        if d_embed is None:
            raise ValueError("d_embed must be specified for SHUFFLED_RANKPE")
        return RankEmbedWrapper(env, d_embed=d_embed)
    if exp_condition is Condition.SHUFFLED_DISTPE:
        if d_embed is None:
            raise ValueError("d_embed must be specified for SHUFFLED_DISTPE")
        return DistanceEmbedWrapper(env, d_embed=d_embed)
    if exp_condition is Condition.SHUFFLED_ROPE:
        return RotaryEmbedWrapper(env, rotate_dim=d_embed)
    return env


def embed_spec_for(exp_condition: Condition, cfg: Dict[str, Any], d_embed: Optional[int],
                   validate: bool = True) -> EmbedSpec:
    """The fused-embedding description the wrappers would configure for this condition."""
    import numpy as np
    import torch

    from .._lib import EMBED_DIST, EMBED_RANK, EMBED_ROPE
    from ..utils.defaults import max_dist

    obs = resolve_config(cfg)["observation"]
    N, F = int(obs["vehicles_count"]), len(obs["features"])
    if exp_condition is Condition.SHUFFLED_ROPE:
        rd = d_embed or (F - (F % 2))
        if rd % 2 != 0 or rd > F:
            raise ValueError(f"rotate_dim must be even and ≤ {F}; got {rd}")
        return EmbedSpec(EMBED_ROPE, rd, rope_inv_freq(rd, max_dist()), max_dist(), True, 0)
    if exp_condition is Condition.SHUFFLED_DISTPE:
        if d_embed is None:
            raise ValueError("d_embed must be specified for SHUFFLED_DISTPE")
        if d_embed % 2 != 0:
            raise ValueError(f"DistanceEmbedWrapper requires even d_embed; got {d_embed}")
        return EmbedSpec(EMBED_DIST, d_embed, dist_freqs(d_embed, max_dist()).numpy(), max_dist(), True, 0)
    if exp_condition is Condition.SHUFFLED_RANKPE:
        if d_embed is None:
            raise ValueError("d_embed must be specified for SHUFFLED_RANKPE")
        table = torch.nn.Embedding(N, d_embed)
        table.weight.data.uniform_(-0.05, 0.05)
        return EmbedSpec(EMBED_RANK, d_embed, torch.tanh(table.weight.detach()).numpy(), max_dist(), True, 0)
    return EmbedSpec()


def make_vec_env(exp_condition: Condition, base_cfg: Dict[str, Any], d_embed: Optional[int] = None,
                 env_overrides: Dict[str, Any] = {}, num_envs: int = 4096, device: Any = "cuda", seed: int = 0,
                 env_id_base: int = 0, autoreset: bool = True, strict_d_embed: bool = True) -> HighwayVecEnv:
    """``num_envs`` lock-step envs with the condition's embedding fused into the step kernel.

    ``strict_d_embed=False`` skips ``make_env``'s "d_embed ≤ feature count" gate for DistPE, which the
    reference only enforces in the factory -- ``DistanceEmbedWrapper`` itself accepts any even
    ``d_embed`` (SURVEY.md F4; ``visualize.py:147-152`` builds it directly).
    """
    if strict_d_embed:
        cfg = _resolve(exp_condition, base_cfg, d_embed, env_overrides)
    else:
        cfg = _resolve(exp_condition, base_cfg, None, env_overrides)
    spec = embed_spec_for(exp_condition, cfg, d_embed)
    return HighwayVecEnv(cfg, num_envs, device=device, embed=spec, autoreset=autoreset, env_id_base=env_id_base,
                         seed=seed)
