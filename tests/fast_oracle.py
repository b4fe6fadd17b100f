"""highway-fast-v0 on the fp64 oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``oracle/highway_oracle.c`` restates highway-v0, whose ``Road.step`` tests every pair (i, j), i < j.  highway-fast-v0
(``HighwayEnvFast``, DESIGN.md Appendix C) switches collision checks off on every uncontrolled vehicle, so only the
pairs of the ego (i = 0) are tested, and changes nothing else but its defaults.  This module states exactly that
difference on top of the unchanged oracle:

* the oracle's C source is compiled a second time with the bound of that one loop changed from ``i < e->V`` to
  ``i < 1`` (into a temporary directory, keyed by a hash of the source);
* ``highway`` is a second instance of ``oracle/highway.py`` bound to that library, whose ``cfg_from_dict`` first
  applies ``HighwayEnvFast.default_config()``'s entries under the user's keys (the oracle's own knows highway-v0's
  defaults only).  It is a drop-in for ``oracle.highway`` wherever a fast env is compared.

Parity unpinned, as for the whole simulator (DESIGN.md §4).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import importlib.util
import os
import subprocess
import tempfile
from typing import Any, Dict

from oracle import highway as v0

FAST = "highway-fast-v0"
# HighwayEnvFast.default_config(): HighwayEnv's, updated with these (highway-env 1.10.1)
FAST_DEFAULTS: Dict[str, Any] = {"simulation_frequency": 5, "lanes_count": 3, "vehicles_count": 20, "duration": 30,
                                 "ego_spacing": 1.5}
_ALL_PAIRS = "for (int i = 0; i < e->V; ++i)\n            for (int j = i + 1; j < e->V; ++j) handle_collisions(e, i, j, dt);"
_EGO_PAIRS = "for (int i = 0; i < 1; ++i)\n            for (int j = i + 1; j < e->V; ++j) handle_collisions(e, i, j, dt);"


def fast_config(cfg: Dict[str, Any]) -> Dict[str, Any]:
    """``cfg`` over HighwayEnvFast's defaults (a shallow update, as ``configure`` does)"""
    full = dict(FAST_DEFAULTS)
    full.update(cfg)
    return full


def _build() -> str:
    with open(v0._SRC) as f:
        src = f.read()
    if src.count(_ALL_PAIRS) != 1:
        raise RuntimeError("oracle/highway_oracle.c: the pair loop of Road.step was not found exactly once")
    src = src.replace(_ALL_PAIRS, _EGO_PAIRS)
    with open(os.path.join(v0._HERE, "highway_oracle.h")) as f:
        tag = hashlib.sha256((src + f.read()).encode()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"hrp_fast_oracle_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    lib = os.path.join(out_dir, f"libhighway_oracle_fast_{tag}.so")
    if not os.path.exists(lib):
        c_file = os.path.join(out_dir, f"highway_oracle_fast_{tag}_{os.getpid()}.c")
        with open(c_file, "w") as f:
            f.write(src)
        tmp = f"{lib}.{os.getpid()}.tmp"
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-I", v0._HERE, "-o", tmp, c_file, "-lm"])
        os.replace(tmp, lib)
        os.remove(c_file)
    return lib


def _load():
    spec = importlib.util.spec_from_file_location("oracle_highway_fast", v0.__file__)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod._lib = mod._bind(C.CDLL(_build()))
    v0_cfg_from_dict = mod.cfg_from_dict
    mod.cfg_from_dict = lambda cfg: v0_cfg_from_dict(fast_config(cfg))
    return mod


highway = _load()


def oracle_module(cfg: Dict[str, Any]):
    """the oracle module that restates ``cfg``'s env id"""
    return highway if cfg.get("gym_id", "highway-v0") == FAST else v0
