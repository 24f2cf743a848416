"""Host-side mirror of the reference's forest-fire generator (/root/reference/src/DynamicArea.jl),
running the automaton on the device and feeding the coverage cell store directly -- no xlsx
hand-off (SURVEY.md 8f-3).

The reference script draws from Julia's global RNG; here every draw is a counter-based Philox
uniform keyed by (seed, step, cell, neighbour), so host and device restatements agree bit for bit.
"""
from __future__ import annotations

import math

import numpy as np

from .engine import CoverageEngine

EMPTY, TREE, FIRE = 0, 1, 2  # src/DynamicArea.jl:17


class ForestFire:
    """Parameters as in src/DynamicArea.jl:5-22,47-48; `engine` holds the CA state and the cell store."""

    def __init__(self, engine: CoverageEngine, dx=5.0, dy=5.0, X=500.0, Y=500.0, x_start1=200.0, x_start2=300.0,
                 y_start1=345.0, y_start2=355.0, forest_density=0.7, prob_spread=0.5, wind_speed=4.0,
                 wind_direction=math.radians(270.0), seed=0, push_initial=True):
        self.engine = engine
        self.dx, self.dy = float(dx), float(dy)
        self.nx, self.ny = int(round(X / dx)), int(round(Y / dy))
        self.prob_spread, self.wind_speed, self.wind_direction = prob_spread, wind_speed, wind_direction
        self.seed = int(seed)
        self.t = 0
        rng = np.random.default_rng(np.random.PCG64(seed))
        # grid[i, j]: TREE with probability forest_density, else EMPTY (:26-33); i outer, j inner
        grid = np.where(rng.random((self.nx, self.ny)) < forest_density, TREE, EMPTY).astype(np.uint8)
        i0, i1 = int(round(x_start1 / dx)), int(round(x_start2 / dx))
        j0, j1 = int(round(y_start1 / dy)), int(round(y_start2 / dy))
        grid[i0 - 1:i1, j0 - 1:j1] = FIRE  # :35 (1-based inclusive ranges)
        self.initial_grid = grid
        engine.fire_init(grid.T.ravel(), self.nx, self.ny, self.dx, self.dy, push_initial=push_initial)

    def step(self, append: bool = True) -> int:
        """One update_grid() (:52-72): returns the number of list entries pushed."""
        self.t += 1
        return self.engine.fire_step(self.wind_speed, self.wind_direction, self.prob_spread, self.seed, self.t,
                                     append=append)

    def run_horizon(self, x_start, fire_steps, **kw):
        """CoverageEngine.run_horizon_fire on this fire: timestep t runs fire_steps[t-1] of this fire's steps before
        its rmvCoveredPOI, continuing the step numbers of step(), so that later step() calls continue the same stream.
        kw: run_horizon's S, spread, n_iter, granularity, seed, boxes, h_focus, h_max."""
        fire_steps = np.ascontiguousarray(fire_steps, dtype=np.int64).ravel()
        out = self.engine.run_horizon_fire(x_start, fire_steps, self.wind_speed, self.wind_direction,
                                           self.prob_spread, self.seed, self.t + 1, **kw)
        self.t += int(fire_steps.sum())
        return out

    def run_horizon_ensemble(self, x_starts, fire_steps, winds=None, fire_seed_stride: int = 1, **kw):
        """CoverageEngine.run_horizon_fire_ensemble from this fire's current state: E scenarios, each with its own
        starting swarm (x_starts (E, 3N)), wind (winds (E, 3) or (3,); None: this fire's wind for every scenario) and
        fire seed self.seed + e * fire_seed_stride, all continuing at step self.t + 1, so that scenario 0 is this fire's
        own run_horizon.  Unlike run_horizon it leaves self.t as it is: the engine's fire has not moved.
        kw: run_horizon_fire_ensemble's S, spread, n_iter, granularity, seed, boxes, h_focus, h_max, want_cells,
        want_states."""
        if winds is None:
            winds = (self.wind_speed, self.wind_direction, self.prob_spread)
        return self.engine.run_horizon_fire_ensemble(x_starts, fire_steps, winds, self.seed, self.t + 1,
                                                     fire_seed_stride=fire_seed_stride, **kw)

    def grid(self) -> np.ndarray:
        """Current state as grid[i-1, j-1]."""
        return self.engine.fire_state().reshape(self.ny, self.nx).T
