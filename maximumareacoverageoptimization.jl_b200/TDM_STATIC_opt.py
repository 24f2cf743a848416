"""Host-side mirror of the reference module `TDM_STATIC_opt`
(/root/reference/src/TDM_STATIC_opt.jl): `createObjective(cells, N, r_max)` returns the closure
`AreaMaxObjective(x)` with the reference's value semantics; the closure additionally exposes
`.batch(X)` (a whole MADS poll set in one cov_eval_batch call) and `.fuse(constraints)`.
`optimize(...)` is in mads.py (the batched poll driver) and re-exported here.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .CellFunctions import Cells
from .AreaCoverageCalculation import PointList, ResidentList


class AreaMaxObjective:
    """src/TDM_STATIC_opt.jl:83-98:  -calculateArea(x, cells.points_of_interest)
    + 1e5 * sum_i abs(x[i+2N] - r_max[i])."""

    def __init__(self, cells, N: int, r_max):
        self.cells = cells
        self.N = int(N)
        self.r_max = r_max  # captured by reference, like the Julia closure
        self._fused = {}

    def _resident(self) -> ResidentList:
        c = self.cells
        if isinstance(c, Cells):
            return c.resident()
        if isinstance(c, ResidentList):
            return c
        if not hasattr(self, "_own"):
            self._own = ResidentList(PointList.infer(c))
        return self._own

    def fuse(self, constraints):
        """Fold extreme constraints that carry a `.fuse` description (create_cons3/7/8, cons1) into
        this objective's kernel launch; returns the ones that stay host callables."""
        rest = []
        fused = {}
        for c in constraints:
            f = getattr(c, "fuse", None)
            if f is None:
                rest.append(c)
            else:
                fused.update(f)
        self._fused = fused
        return rest

    def native_solver(self, constraints):
        """A callable (x0, n_iter, granularity, seed) -> (x, objective, stats) running cov_mads_solve with these
        extreme constraints fused, or None when a constraint cannot be fused."""
        if self.fuse(constraints):
            return None
        res, eng = self._engine()
        return eng.mads_solve

    def native_batch_solver(self, constraints):
        """A callable (X0, n_iter, granularity, seed) -> (X, objectives, stats) running cov_mads_solve_batch (S solves
        in one launch, solve k seeded seed + k) with these extreme constraints fused, or None when a constraint cannot
        be fused."""
        if self.fuse(constraints):
            return None
        res, eng = self._engine()
        return eng.mads_solve_batch

    def _engine(self):
        res = self._resident()
        eng = res.sync()
        r = np.ascontiguousarray(self.r_max, dtype=np.float64).ravel()
        # the engine is shared (other objectives on the same cells, calculateArea, constraints): the token of
        # whoever configured it last lives on the engine and is cleared by every set_params()
        key = (id(self), r.tobytes(), id(self._fused))
        if eng.param_owner != key or eng.N != self.N:
            eng.set_params(self.N, r, 1e5, **self._fused)
            eng.set_option(_lib.OPT_PROGRESSIVE_INDEX, 0)
            eng.param_owner = key
        return res, eng

    def batch(self, X, want_feasible=False, granularity=1.0):
        """Objective of every row of X (B x 3N).  With want_feasible also the fused extreme
        constraints' verdicts.  An int16 / int32 X holds MESH INDICES (candidate = q * granularity, the MADS mesh of
        src/TDM_STATIC_opt.jl:131-137) and a float32 X values: they travel packed (cov_eval_batch_packed) and are
        widened to Float64 on the device."""
        res, eng = self._engine()
        if isinstance(X, np.ndarray) and X.dtype in (np.int16, np.int32, np.float32):
            out = eng.eval_batch_packed(X.reshape(-1, 3 * self.N), granularity, want_count=False,
                                        want_feasible=want_feasible)
            return (out["obj"], out["feasible"].astype(bool)) if want_feasible else out["obj"]
        X = np.ascontiguousarray(X, dtype=np.float64).reshape(-1, 3 * self.N)
        # (non-dyadic weights, where the Float64 sum depends on the list order, are replayed in list order on the
        # device by the library's ordered kernel: nothing special here)
        out = eng.eval_batch(X, want_count=False, want_feasible=want_feasible)
        if want_feasible:
            return out["obj"], out["feasible"].astype(bool)
        return out["obj"]

    def __call__(self, x) -> float:
        res, eng = self._engine()
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        return eng.eval_one(x)


def createObjective(cells, N, r_max) -> AreaMaxObjective:
    """src/TDM_STATIC_opt.jl:82-100."""
    return AreaMaxObjective(cells, N, r_max)


class RegionObjective(AreaMaxObjective):
    """The grid-free static objective: -A(x) + 1e5 * sum_i abs(x[i+2N] - r_max[i]) with A(x) the exact area of
    (union of the discs of x) n region \\ (union of the covered discs) -- the limit of AreaMaxObjective's value in the
    static environment as the cells shrink (cov_eval_region_batch).  The same closure shape as AreaMaxObjective:
    `__call__`, `.batch`, `.fuse`, `.native_batch_solver` (cov_mads_solve_batch_region); cov_mads_solve has no region
    form, so `native_solver` is None and mads.optimize polls from Python."""

    def __init__(self, region, covered, N: int, r_max, engine=None):
        super().__init__(None, N, r_max)
        self.region = tuple(float(v) for v in region)  # (x_lo, y_lo, x_hi, y_hi)
        self.covered = np.array(np.zeros((0, 3)) if covered is None else covered, dtype=np.float64).reshape(-1, 3)
        self._eng = engine
        self._own_engine = engine is None

    def _engine(self):
        from .engine import CoverageEngine
        if self._eng is None:
            self._eng = CoverageEngine(0)
        eng = self._eng
        r = np.ascontiguousarray(self.r_max, dtype=np.float64).ravel()
        key = (id(self), r.tobytes(), id(self._fused))
        if eng.param_owner != key or eng.N != self.N:
            eng.set_params(self.N, r, 1e5, **self._fused)
            eng.set_region(*self.region, self.covered)  # the region is the objective's: set with its parameters
            eng.param_owner = key
        return None, eng

    def native_solver(self, constraints):
        return None

    def native_batch_solver(self, constraints):
        if self.fuse(constraints):
            return None
        return self._engine()[1].mads_solve_batch_region

    def batch(self, X, want_feasible=False, granularity=1.0):
        eng = self._engine()[1]
        X = np.ascontiguousarray(X, dtype=np.float64).reshape(-1, 3 * self.N)
        out = eng.eval_region_batch(X, want_area=False, want_feasible=want_feasible)
        return (out["obj"], out["feasible"].astype(bool)) if want_feasible else out["obj"]

    def __call__(self, x) -> float:
        return float(self.batch(np.ravel(x))[0])

    def close(self):
        if self._own_engine and self._eng is not None:
            self._eng.close()
            self._eng = None


def createRegionObjective(region, covered, N, r_max, engine=None) -> RegionObjective:
    """The grid-free static objective on the domain region = (x_lo, y_lo, x_hi, y_hi) with the discs `covered`
    (M x 3 rows x, y, R) already covered; engine: a CoverageEngine to run on (default: one of its own)."""
    return RegionObjective(region, covered, N, r_max, engine)


def optimize(input, obj, cons_ext, cons_prog, N_iter, **kw):
    """src/TDM_STATIC_opt.jl:118-222 -- see mads.optimize."""
    from .mads import optimize as _opt
    return _opt(input, obj, cons_ext, cons_prog, N_iter, **kw)


def optimize_multistart(inputs, obj, cons_ext, cons_prog, N_iter, **kw):
    """Several solves in lockstep, one objective launch per iteration for all of them -- see mads.optimize_multistart."""
    from .mads import optimize_multistart as _opt
    return _opt(inputs, obj, cons_ext, cons_prog, N_iter, **kw)
