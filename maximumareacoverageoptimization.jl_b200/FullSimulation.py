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


H_FOCUS = 15.0  # the altitude the r_max rule looks for (src/FullSimulation.jl:66)


def _boxes(p: SimulationParameters) -> np.ndarray:
    """The high-interest rectangles as K x 4 rows x_LB, x_UB, y_LB, y_UB."""
    return np.stack([np.asarray(v, dtype=np.float64).ravel() for v in (p.x_LB, p.x_UB, p.y_LB, p.y_UB)], axis=1)


def apply_r_max_rule(drone_locs, r_max, N: int, p: SimulationParameters, t_half: float):
    """src/FullSimulation.jl:65-76, in place on r_max: a UAV flying at H_FOCUS keeps the focus radius near a
    high-interest rectangle (within h_max * tan(FOV/2) of it) and gets the h_max radius elsewhere."""
    xl, xu, yl, yu = _boxes(p).T
    for i in range(N):
        if abs(H_FOCUS - drone_locs[i + 2 * N] / t_half) < 1:
            m = p.h_max * t_half
            check = ((drone_locs[i] < xu + m) & (drone_locs[i] > xl - m) &
                     (drone_locs[i + N] < yu + m) & (drone_locs[i + N] > yl - m))
            r_max[i] = H_FOCUS * t_half if check.any() else p.h_max * t_half


def run_simulation(cells, starting_circles, cons_ext, cons_prog, N, r_max, params: SimulationParameters,
                   Nt_sim: int | None = None, objective: str = "grid", covered_pb: list | None = None,
                   starts: int | None = None, spread: float = 3.0, list_order: bool = False):
    """Returns (single_input_pb, single_output_pb, runtime_data_MADS, objective_pb).  objective: "grid" (the
    reference's) or "region"; with "region", covered_pb (if given) receives the covered set (M x 3 rows x, y, R) each
    timestep's objective was built on.

    starts=S runs the whole horizon on the device in one call (CoverageEngine.run_horizon): per timestep S MADS
    solves, from the swarm and from S - 1 copies of it moved by N(0, spread^2) metres in x and y, and the best result
    becomes the next swarm.  The grid objective only, with constraints that all fuse; runtime_data_MADS then holds the
    device time of each timestep.  The dynamic environment appends update_POI's rows inside the same call
    (CoverageEngine.run_horizon_points) and leaves cells as the host loop does.  list_order=True lets that call run
    on a store whose area depends on the list order (a high-interest rectangle where the fire is gives its entries
    the non-dyadic weight (h_max tan(FOV/2))^2 pi); without it such a store raises COV_ERR_STATE."""
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
    if starts is not None:
        if objective != "grid":
            raise ValueError("starts= runs the grid objective only")
        if p.environment_type == "dynamic" and getattr(cells, "fire_rows", None) is None:
            raise ValueError("starts= with the dynamic environment needs cells with fire_rows (initialise_POI)")
        return _run_horizon(cells, pre, cons_ext, N, r_max, p, steps, int(starts), spread, t_half, d_lim, list_order)
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
            apply_r_max_rule(drone_locs, r_max, N, p, t_half)
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


def _run_horizon(cells, pre, cons_ext, N, r_max, p, steps, S, spread, t_half, d_lim, list_order=False):
    """run_simulation(starts=S): the loop above with S solves per timestep, in one cov_run_horizon call."""
    from .mads import _flatten_constraints
    boxes = _boxes(p)
    if not len(boxes):
        raise ValueError("starts= needs at least one high-interest rectangle")
    obj = TDM_STATIC_opt.createObjective(cells, N, r_max)
    if obj.native_batch_solver(_flatten_constraints([cons_ext, create_cons3(pre, p.FOV, d_lim)])) is None:
        raise ValueError("starts= needs constraints that all fuse into the objective's launch")
    res, eng = obj._engine()  # the store synced, the parameters of timestep 1's solves (cons3 from pre) set
    kw = dict(S=S, spread=spread, n_iter=p.N_iter, granularity=1.0, seed=0 if p.seed is None else p.seed,
              boxes=boxes, h_focus=H_FOCUS, h_max=p.h_max, list_order=list_order)
    if p.environment_type == "dynamic":
        appends = CellFunctions.update_POI_schedule(cells, steps)
        X, objs, _, step_ms, last = eng.run_horizon_points(pre, appends, **kw)
        # the host list as update_POI and rmvCoveredPOI leave it: an entry appended at timestep ta (1 for the
        # initial list) is gone iff its cell lost entries at ta or later
        ta = np.concatenate([np.ones(len(res.points), dtype=np.int64)] +
                            [np.full(len(a), t, dtype=np.int64) for t, a in enumerate(appends, start=1)])
        for a in appends:
            if len(a):
                res.points.append(a)
                cells.fire_point_xy_ccordinates.extend(q[:2].copy() for q in a)
        res.points.keep(last[res.points.cell_index()] < ta)
    else:
        X, objs, _, step_ms = eng.run_horizon(pre, steps, **kw)
        # the host list after every rmvCoveredPOI: the entries whose cell still holds some
        res.points.keep(eng.grid_cells()[res.cell_index()] > 0)
    res.mark_synced()
    for t in range(2, steps + 1):  # the caller's r_max as the host loop leaves it
        apply_r_max_rule(X[t - 2], r_max, N, p, t_half)
    inputs = [pre.copy()] + [X[t].copy() for t in range(steps - 1)]
    return inputs, [x.copy() for x in X], [float(ms) / 1e3 for ms in step_ms], [float(v) for v in objs]


def run_simulation_region(cells, starting_circles, cons_ext, N, r_max, params: SimulationParameters,
                          Nt_sim: int | None = None, starts: int = 1, spread: float = 3.0, covered_pb: list | None = None):
    """run_simulation(objective="region") with S = starts solves per timestep, the whole horizon on the device in one
    cov_run_horizon_region call (CoverageEngine.run_horizon_region): the domain is the cell lattice's rectangle, the
    covered set starts empty and every timestep appends the current swarm's discs to it.  Static environment, with
    constraints that all fuse.  Returns run_simulation's 4-tuple (runtime_data_MADS: the device time of each timestep)
    and leaves the caller's r_max as the host loop does; covered_pb (if given) receives the covered set (M x 3 rows
    x, y, R) each timestep's objective was built on.  cells is only read."""
    from .mads import _flatten_constraints
    p = params
    if p.environment_type != "static":
        raise ValueError("the region objective has no dynamic form: its points are not cells")
    boxes = _boxes(p)
    if not len(boxes):
        raise ValueError("starts= needs at least one high-interest rectangle")
    t_half = math.tan(p.FOV / 2)
    pre = np.ascontiguousarray(starting_circles if not hasattr(starting_circles[0], "x")
                               else ACC.make_MADS(starting_circles), dtype=np.float64)
    r_max = np.ascontiguousarray(r_max, dtype=np.float64)
    steps = p.Nt_sim if Nt_sim is None else Nt_sim
    pl = cells.points_of_interest
    region = (0.0, 0.0, pl.nx * pl.dx, pl.ny * pl.dy)
    obj = TDM_STATIC_opt.createRegionObjective(region, None, N, r_max.copy())
    try:
        cons = _flatten_constraints([cons_ext, create_cons3(pre, p.FOV, p.d_lim * np.ones(N))])
        if obj.native_batch_solver(cons) is None:
            raise ValueError("starts= needs constraints that all fuse into the objective's launch")
        _, eng = obj._engine()  # the empty region and the parameters of timestep 1's solves (cons3 from pre) set
        X, objs, _, step_ms = eng.run_horizon_region(pre, steps, S=int(starts), spread=spread, n_iter=p.N_iter,
                                                     granularity=1.0, seed=0 if p.seed is None else p.seed,
                                                     boxes=boxes, h_focus=H_FOCUS, h_max=p.h_max)
    finally:
        obj.close()
    inputs = [pre.copy()] + [X[t].copy() for t in range(steps - 1)]
    if covered_pb is not None:  # timestep t's objective: the swarms of timesteps 1 .. t before their solves
        for t in range(1, steps + 1):
            covered_pb.append(np.concatenate([x.reshape(3, N).T for x in inputs[:t]]))
    for t in range(2, steps + 1):  # the caller's r_max as the host loop leaves it
        apply_r_max_rule(X[t - 2], r_max, N, p, t_half)
    return inputs, [x.copy() for x in X], [float(ms) / 1e3 for ms in step_ms], [float(v) for v in objs]


def run_simulation_ensemble(cells, starting_swarms, cons_ext, N, r_max, params: SimulationParameters,
                            Nt_sim: int | None = None, starts: int = 1, spread: float = 3.0, list_order: bool = False):
    """run_simulation(starts=S) from E starting swarms at once, in one cov_run_horizon_ensemble call (static
    environment) or one cov_run_horizon_points_ensemble call (dynamic environment, on cells with fire_rows: every
    scenario appends update_POI's rows): scenario e is run_simulation(starts=S) from starting_swarms[e] with
    params.seed + e * Nt_sim * S (base seed 0 when params.seed is None).  Returns a list of E tuples (single_input_pb,
    single_output_pb, runtime_data_MADS, objective_pb), each what run_simulation(starts=S) returns for that scenario,
    except that runtime_data_MADS holds the device time of each timestep of the whole ensemble.  Unlike run_simulation,
    cells (its point list and the store on the device) and the caller's r_max are left untouched.  list_order: as for
    run_simulation."""
    from .mads import _flatten_constraints
    p = params
    if p.environment_type not in ("static", "dynamic"):
        raise ValueError("environment_type must be 'static' or 'dynamic'")
    dynamic = p.environment_type == "dynamic"
    if dynamic and getattr(cells, "fire_rows", None) is None:
        raise ValueError("the dynamic environment needs cells with fire_rows (initialise_POI)")
    pres = [np.ascontiguousarray(s if not hasattr(s[0], "x") else ACC.make_MADS(s), dtype=np.float64)
            for s in starting_swarms]
    if not pres:
        raise ValueError("starting_swarms must hold at least one swarm")
    d_lim = p.d_lim * np.ones(N)
    steps = p.Nt_sim if Nt_sim is None else Nt_sim
    S = int(starts)
    if not len(_boxes(p)):
        raise ValueError("starts= needs at least one high-interest rectangle")
    obj = TDM_STATIC_opt.createObjective(cells, N, np.array(r_max, dtype=np.float64))
    for pre in pres:  # the last one's cons3 stays set; every timestep replaces the previous swarm on the device
        if obj.native_batch_solver(_flatten_constraints([cons_ext, create_cons3(pre, p.FOV, d_lim)])) is None:
            raise ValueError("starts= needs constraints that all fuse into the objective's launch")
    _, eng = obj._engine()
    kw = dict(S=S, spread=spread, n_iter=p.N_iter, granularity=1.0, seed=0 if p.seed is None else p.seed,
              boxes=_boxes(p), h_focus=H_FOCUS, h_max=p.h_max, list_order=list_order)
    if dynamic:
        schedule = CellFunctions.update_POI_schedule(cells, steps)
        X, objs, _, step_ms = eng.run_horizon_points_ensemble(np.stack(pres), [schedule], **kw)
    else:
        X, objs, _, step_ms = eng.run_horizon_ensemble(np.stack(pres), steps, **kw)
    runtime = [float(ms) / 1e3 for ms in step_ms]
    return [([pre.copy()] + [Xe[t].copy() for t in range(steps - 1)], [x.copy() for x in Xe], list(runtime),
             [float(v) for v in oe]) for pre, Xe, oe in zip(pres, X, objs)]
