"""tests/grid_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

fp64, sequential restatement of highway-env 1.10.1 ``OccupancyGridObservation.observe`` (``absolute=False``,
``as_image=False``) as DESIGN.md §3.1 and Appendix B state it: the contract the grid epilogue of the step kernel
follows.  PARITY UNPINNED, like the Kinematics restatement: upstream cannot be imported here (DESIGN.md §4).

Written literally: the vehicles in reverse list order (upstream's ``df[::-1]``, so the lowest index ends up owning a
shared cell), an explicit ``arange`` for the road layer, plain Python floats (IEEE fp64, no fused multiply-add).

Every ``floor`` that yields a cell index is a keyed decision, as the simulator oracle's ``dec()`` is: ``("veh", k,
axis)`` for vehicle k and ``("road", lane, i, axis)`` for waypoint i of a lane, with margin = distance in metres to the
nearer cell boundary.  ``record_below`` lists the decisions taken by less than that margin in ``marginal``; a key in
``forced`` is decided the other way (the neighbouring cell across the nearer boundary).  ``either_branch`` uses them to
judge the fp32 kernel, whose headings (and so rotated positions) differ from fp64 in the last bits.
"""
from __future__ import annotations

import itertools
import math
from typing import Any, Dict, Optional, Sequence

import numpy as np

DEFAULT_RANGE = {"vx": [-80.0, 80.0], "vy": [-80.0, 80.0]}   # +-2 Vehicle.MAX_SPEED
ROAD_LENGTH = 10000.0
LANE_WIDTH = 4.0
LANE_PERCEPTION = 100.0


def lmap(v, x, y):
    """utils.lmap: y[0] + (v - x[0]) * (y[1] - y[0]) / (x[1] - x[0])"""
    return y[0] + (v - x[0]) * (y[1] - y[0]) / (x[1] - x[0])


class GridOracle:
    def __init__(self, features: Sequence[str] = ("presence", "vx", "vy", "on_road"),
                 grid_size=((-27.5, 27.5), (-27.5, 27.5)), grid_step=(5.0, 5.0),
                 features_range: Optional[Dict[str, Any]] = None, align_to_vehicle_axes: bool = False,
                 clip: bool = True, lanes: int = 4):
        self.features = list(features)
        self.size = [[float(a), float(b)] for a, b in grid_size]
        self.step = [float(s) for s in grid_step]
        self.ranges = {k: [float(v[0]), float(v[1])] for k, v in (features_range or DEFAULT_RANGE).items()}
        self.align = bool(align_to_vehicle_axes)
        self.clip = bool(clip)
        self.lanes = int(lanes)
        self.W = int(math.floor((self.size[0][1] - self.size[0][0]) / self.step[0]))
        self.H = int(math.floor((self.size[1][1] - self.size[1][0]) / self.step[1]))
        self.record_below = 0.0
        self.forced: set = set()
        self.marginal: Dict[Any, float] = {}

    @property
    def shape(self):
        return (len(self.features), self.W, self.H)

    # ---- keyed floor and pos_to_index
    def _floor(self, key, t: float, step: float) -> int:
        f = math.floor(t)
        below, above = (t - f) * step, (f + 1 - t) * step
        if min(below, above) < self.record_below:
            self.marginal[key] = min(below, above)
        if key in self.forced:
            return f - 1 if below <= above else f + 1
        return f

    def _cell(self, key, px: float, py: float, c: float, s: float):
        if self.align:
            px, py = c * px + s * py, (-s) * px + c * py
        ix = self._floor(key + (0,), (px - self.size[0][0]) / self.step[0], self.step[0])
        iy = self._floor(key + (1,), (py - self.size[1][0]) / self.step[1], self.step[1])
        return (ix, iy) if 0 <= ix < self.W and 0 <= iy < self.H else None

    # ---- observe
    def observe(self, x, y, heading, speed):
        """Grid [F, W, H] float32 and cell vehicles [W * H] int32 (-1: no vehicle) of one env; vehicle 0 is the ego."""
        V = len(x)
        self.marginal = {}
        x, y = [float(v) for v in x], [float(v) for v in y]
        heading, speed = [float(v) for v in heading], [float(v) for v in speed]
        c, s = math.cos(heading[0]), math.sin(heading[0])

        def to_dict(k):   # Vehicle.to_dict(ego), then normalize() over features_range
            vx0, vy0 = speed[0] * math.cos(heading[0]), speed[0] * math.sin(heading[0])
            d = {"presence": 1.0, "x": x[k] - x[0], "y": y[k] - y[0],
                 "vx": speed[k] * math.cos(heading[k]) - vx0, "vy": speed[k] * math.sin(heading[k]) - vy0,
                 "heading": heading[k], "cos_h": math.cos(heading[k]), "sin_h": math.sin(heading[k])}
            for f, r in self.ranges.items():
                if f in d:
                    d[f] = lmap(d[f], r, [-1.0, 1.0])
            return d

        def position(d):
            px, py = d["x"], d["y"]
            if "x" in self.ranges:
                px = lmap(px, [-1.0, 1.0], self.ranges["x"])
            if "y" in self.ranges:
                py = lmap(py, [-1.0, 1.0], self.ranges["y"])
            return px, py

        grid = np.full(self.shape, np.nan, dtype=np.float64)
        cells = np.full((self.W, self.H), -1, dtype=np.int32)
        for k in reversed(range(V)):
            cell = self._cell(("veh", k), *position(to_dict(k)), c, s)
            if cell is not None:
                cells[cell] = k
        for layer, feature in enumerate(self.features):
            if feature == "on_road":
                self._road_layer(grid, layer, x[0], y[0], c, s)
                continue
            for k in reversed(range(V)):
                d = to_dict(k)
                cell = self._cell(("veh", k), *position(d), c, s)
                if cell is not None:
                    grid[(layer,) + cell] = d[feature]
        if self.clip:
            grid = np.clip(grid, -1, 1)
        return np.nan_to_num(grid).astype(np.float32), cells.reshape(-1)

    def _road_layer(self, grid, layer, ex, ey, c, s):
        """fill_road_layer_by_lanes: lane L is the straight line y = 4 L, x in [0, ROAD_LENGTH]"""
        step = min(self.step)
        start, stop = ex - LANE_PERCEPTION, ex + LANE_PERCEPTION
        n = int(math.ceil((stop - start) / step))   # len(np.arange(start, stop, step))
        for L in range(self.lanes):
            for i in range(n):
                w = min(max(start + i * step, 0.0), ROAD_LENGTH)   # np.clip(waypoints, 0, lane.length)
                cell = self._cell(("road", L, i), w - ex, LANE_WIDTH * L - ey, c, s)
                if cell is not None:
                    grid[(layer,) + cell] = 1.0


def oracle_for(obs_cfg: Dict[str, Any], lanes: int) -> GridOracle:
    """A GridOracle from a resolved OccupancyGrid observation dict."""
    return GridOracle(obs_cfg["features"], obs_cfg["grid_size"], obs_cfg["grid_step"], obs_cfg.get("features_range"),
                      obs_cfg.get("align_to_vehicle_axes", False), obs_cfg.get("clip", True), lanes)


def matches(o: GridOracle, grid, cells, want_grid, want_cells, tol: float) -> bool:
    return bool(np.array_equal(cells, want_cells) and np.max(np.abs(grid - want_grid), initial=0.0) <= tol)


def either_branch(o: GridOracle, state, grid, cells, tol: float, margin: float = 1e-3, max_flips: int = 3):
    """None when the kernel's grid / cell vehicles equal the oracle's as computed; else the set of marginal decisions
    (decided by less than ``margin`` metres) under which they do, or False when no set of up to ``max_flips`` does."""
    o.record_below = margin
    o.forced = set()
    want, want_cells = o.observe(*state)
    keys = sorted(o.marginal, key=lambda k: o.marginal[k])
    try:
        if matches(o, grid, cells, want, want_cells, tol):
            return None
        for r in range(1, max_flips + 1):
            for combo in itertools.combinations(keys, r):
                o.forced = set(combo)
                want, want_cells = o.observe(*state)
                if matches(o, grid, cells, want, want_cells, tol):
                    return set(combo)
        return False
    finally:
        o.forced = set()
        o.record_below = 0.0
