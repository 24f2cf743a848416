"""The MADS section of the reference's receding-horizon driver
(/root/reference/src/FullSimulation.jl:42-107, parameters :727-769), on the GPU objective.

Per timestep, exactly as the reference orders it: optional `update_POI` (dynamic fire), remove the
points the UAVs already cover (`rmvCoveredPOI`), the r_max adjustment near the high-interest
rectangle, `create_cons3` from the previous positions, `createObjective`, `optimize`.  The
trajectory side-stack (ALTRO / ORCA, :115-251) is out of scope: the UAVs are taken to reach the
MADS targets, so the next step's `pre_optimized_circles_MADS` is the MADS output.

objective="region" (static environment only) optimises the grid-free static objective instead
(TDM_STATIC_opt.createRegionObjective): the domain is the cell lattice's rectangle, and where rmvCoveredPOI would
remove the cells the previous swarm covers, its discs are appended to the covered set.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

from . import AreaCoverageCalculation as ACC
from . import CellFunctions, TDM_STATIC_opt
from .TDM_Constraints import cons1, create_cons3


@dataclass
class SimulationParameters:
    """src/FullSimulation.jl:727-769."""
    N: int = 5
    tf: float = 20.0
    dt_sim: float = 0.5
    FOV: float = 100 / 180 * math.pi
    h_min: float = 5.0
    h_max: float = 30.0
    d_lim: float = 10.0
    N_iter: int = 100
    environment_type: str = "static"
    x_LB: tuple = (2500.0,)
    x_UB: tuple = (3500.0,)
    y_LB: tuple = (1000.0,)
    y_UB: tuple = (2000.0,)
    seed: int | None = None
    Nt_sim: int = field(init=False)

    def __post_init__(self):
        self.Nt_sim = int(self.tf / self.dt_sim)


def run_simulation(cells, starting_circles, cons_ext, cons_prog, N, r_max, params: SimulationParameters,
                   Nt_sim: int | None = None, objective: str = "grid", covered_pb: list | None = None):
    """Returns (single_input_pb, single_output_pb, runtime_data_MADS, objective_pb).  objective: "grid" (the
    reference's) or "region"; with "region", covered_pb (if given) receives the covered set (M x 3 rows x, y, R) each
    timestep's objective was built on."""
    p = params
    if objective not in ("grid", "region"):
        raise ValueError("objective must be 'grid' or 'region'")
    if objective == "region" and p.environment_type != "static":
        raise ValueError("the region objective has no dynamic form: its points are not cells")
    t_half = math.tan(p.FOV / 2)
    single_input_pb, single_output_pb, runtime_data_MADS, objective_pb = [], [], [], []
    pre = np.ascontiguousarray(starting_circles if not hasattr(starting_circles[0], "x")
                               else ACC.make_MADS(starting_circles), dtype=np.float64)
    r_max = np.ascontiguousarray(r_max, dtype=np.float64)
    d_lim = p.d_lim * np.ones(N)
    steps = p.Nt_sim if Nt_sim is None else Nt_sim
    engine, covered = None, np.zeros((0, 3))
    if objective == "region":
        from .engine import CoverageEngine
        pl = cells.points_of_interest
        region = (0.0, 0.0, pl.nx * pl.dx, pl.ny * pl.dy)
        engine = CoverageEngine(getattr(cells, "device", 0))
    for t in range(1, steps + 1):
        if p.environment_type == "dynamic":
            cells = CellFunctions.update_POI(cells, t)
        drone_locs = pre.copy()
        if objective == "region":
            covered = np.vstack([covered, drone_locs.reshape(3, N).T])
        else:
            cells = CellFunctions.rmvCoveredPOI(cells, drone_locs)
        if t != 1:  # :65-76
            xl, xu, yl, yu = (np.asarray(v, dtype=np.float64) for v in (p.x_LB, p.x_UB, p.y_LB, p.y_UB))
            for i in range(N):
                if abs(15 - drone_locs[i + 2 * N] / t_half) < 1:
                    m = p.h_max * t_half
                    check = ((drone_locs[i] < xu + m) & (drone_locs[i] > xl - m) &
                             (drone_locs[i + N] < yu + m) & (drone_locs[i + N] > yl - m))
                    r_max[i] = 15 * t_half if check.any() else p.h_max * t_half
        cons3 = create_cons3(pre, p.FOV, d_lim)
        if t < 3:
            single_input = drone_locs
        else:
            single_input = single_output_pb[-1]
            if not cons1(single_input) or not cons3(single_input):
                single_input = drone_locs
        if objective == "region":
            area_objective_func = TDM_STATIC_opt.createRegionObjective(region, covered, N, r_max, engine=engine)
            if covered_pb is not None:
                covered_pb.append(covered.copy())
        else:
            area_objective_func = TDM_STATIC_opt.createObjective(cells, N, r_max)
        out, runtime = TDM_STATIC_opt.optimize(single_input, area_objective_func, [cons_ext, cons3], cons_prog,
                                               p.N_iter, seed=None if p.seed is None else p.seed + t)
        runtime_data_MADS.append(runtime)
        single_input_pb.append(np.array(single_input))
        single_output_pb.append(np.array(out))
        objective_pb.append(area_objective_func(out))
        pre = np.array(out)
    if engine is not None:
        engine.close()
    return single_input_pb, single_output_pb, runtime_data_MADS, objective_pb
