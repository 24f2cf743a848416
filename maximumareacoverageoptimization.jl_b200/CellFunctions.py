"""Host-side mirror of the reference module `CellFunctions`
(/root/reference/src/CellFunctions.jl): the cell store `Cells` with `initialise_POI`,
`update_POI`, `rmvCoveredPOI`.  The store lives on the device (libcoverage_cuda's cell store);
the host list is kept alongside because it is user-visible state in the reference.

The reference's dynamic branch is broken as committed (hard-coded Windows path, XLSX not
imported, undefined locals -- SURVEY.md 3.2); this mirror follows its unambiguous intent: the
initial list is rows 1..10 of the fire-point table, and timestep t >= 2 appends row t + 10.
"""
from __future__ import annotations

import math

import numpy as np

from . import AreaCoverageCalculation as ACC
from .AreaCoverageCalculation import PointList, ResidentList
from .engine import TAN_HALF_FOV_DEFAULT


class Cells:
    """src/CellFunctions.jl:5-16 -- `points_of_interest`, `fire_point_xy_ccordinates`."""

    def __init__(self, points_of_interest=None, fire_point_xy_ccordinates=None, device: int = 0):
        self.points_of_interest = points_of_interest if points_of_interest is not None else PointList(
            np.zeros((0, 5)), 100, 100, 5.0, 5.0)
        self.fire_point_xy_ccordinates = fire_point_xy_ccordinates if fire_point_xy_ccordinates is not None else []
        self.device = device
        self._resident = None
        # scenario state the reference reads from Main-scope globals (src/FullSimulation.jl:735-763)
        self.fire_rows = None
        self.high_interest = None  # (x_LB, x_UB, y_LB, y_UB) arrays or None
        self.h_max = 30.0
        self.tan_half_fov = TAN_HALF_FOV_DEFAULT

    def resident(self) -> ResidentList:
        if self._resident is None or self._resident.points is not self.points_of_interest:
            eng = self._resident.engine if self._resident is not None else None
            self._resident = ResidentList(self.points_of_interest, self.device, engine=eng)
        return self._resident

    def close(self):
        if self._resident is not None:
            self._resident.engine.close()
            self._resident = None

    def _reweight(self, pts5: np.ndarray) -> np.ndarray:
        """src/CellFunctions.jl:41-45,68-72: entries strictly inside a high-interest rectangle get
        weight (h_max*tan(FOV/2))^2 * pi."""
        if self.high_interest is None:
            return pts5
        x_LB, x_UB, y_LB, y_UB = (np.atleast_1d(np.asarray(v, dtype=np.float64)) for v in self.high_interest)
        pts5 = pts5.copy()
        x, y = pts5[:, 0:1], pts5[:, 1:2]
        inside = ((x < x_UB) & (x > x_LB) & (y < y_UB) & (y > y_LB)).any(axis=1)
        pts5[inside, 3] = (self.h_max * self.tan_half_fov) ** 2 * math.pi
        return pts5


def initialise_POI(self: Cells, environment_type: str, fire_rows=None, nx=100, ny=100, dx=5.0, dy=5.0,
                   initial_rows: int = 10) -> Cells:
    """src/CellFunctions.jl:20-57.  `fire_rows`: list of (n_k x 5) arrays, one per row of the
    fire-point table (fire_io.load_fire_rows)."""
    if environment_type == "dynamic":
        if fire_rows is None:
            raise ValueError("dynamic environment needs fire_rows (see fire_io.load_fire_rows)")
        self.fire_rows = fire_rows
        rows = [self._reweight(np.asarray(r, dtype=np.float64).reshape(-1, 5)) for r in fire_rows[:initial_rows]]
        data = np.concatenate(rows, axis=0) if rows else np.zeros((0, 5))
        self.points_of_interest = PointList(data, nx, ny, dx, dy)
        self.fire_point_xy_ccordinates = [p[:2].copy() for p in data]
        self._initial_rows = initial_rows
    else:
        # static: createPOI(5.0, 5.0, 100.0, 100.0)  (src/CellFunctions.jl:53)
        self.points_of_interest = ACC.createPOI(5.0, 5.0, 100.0, 100.0)
    return self


def update_POI(self: Cells, t: int) -> Cells:
    """src/CellFunctions.jl:59-79 -- at timestep t != 1 append row t + 10 of the table."""
    if t != 1 and self.fire_rows is not None:
        k = t + getattr(self, "_initial_rows", 10)  # 1-based row number
        if k <= len(self.fire_rows):
            new = self._reweight(np.asarray(self.fire_rows[k - 1], dtype=np.float64).reshape(-1, 5))
            res = self.resident()
            in_sync = res._synced == (id(self.points_of_interest), self.points_of_interest.version)
            self.points_of_interest.append(new)
            self.fire_point_xy_ccordinates.extend(p[:2].copy() for p in new)
            if in_sync:  # append on the device as well instead of re-uploading the whole list
                res.engine.add_points(new)
                res.mark_synced()
    return self


def update_POI_schedule(self: Cells, T: int) -> list:
    """What update_POI appends at timesteps 1 .. T, as T arrays (n_t x 5): nothing at t = 1, then row
    t + initial_rows of the table (reweighted) while rows remain.  The appends of CoverageEngine.run_horizon_points."""
    if self.fire_rows is None:
        raise ValueError("the dynamic schedule needs fire_rows (see initialise_POI)")
    first = getattr(self, "_initial_rows", 10)
    out = []
    for t in range(1, T + 1):
        k = t + first  # 1-based row number
        if t != 1 and k <= len(self.fire_rows):
            out.append(self._reweight(np.asarray(self.fire_rows[k - 1], dtype=np.float64).reshape(-1, 5)))
        else:
            out.append(np.zeros((0, 5)))
    return out


def rmvCoveredPOI(self: Cells, circles) -> Cells:
    """src/CellFunctions.jl:81-108 -- delete every entry covered by the current discs."""
    ACC.rmvCoveredPOI(circles, self.resident())
    return self
