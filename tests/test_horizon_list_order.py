"""COV_OPT_LIST_ORDER_HORIZON: cov_run_horizon, cov_run_horizon_points and their ensembles on stores whose area depends
on the list order (non-dyadic weights: the high-interest weight (h_max tan(FOV/2))^2 pi of update_POI's rectangle).

CPU: what nvcc built for the two list-order kernels, and that the counted inventories around them are unchanged; the
option's constant; the engine keyword puts the option back when the call raises.  GPU: every horizon bit for bit
against the same horizon replayed from single calls on a twin handle (X, objectives, every stats column,
last_removed), both handles alike afterwards (the ordered list included, through 1000 evaluations and one more
non-dyadic entry); every ensemble scenario against the single call; run_simulation and run_simulation_ensemble with
list_order=True; the option on dyadic stores changes nothing; the refusals that stay.
"""
import ctypes as C
import math
import os
import re
import subprocess
import types

import numpy as np
import pytest

from test_horizon import CUOBJDUMP, LIB, REF_BOXES, T_HALF
from test_horizon_dynamic import _params, cell_of, centres, replay, same_handles
from test_horizon_ensemble import _snapshot as _snapshot_static
from test_horizon_points_ensemble import _bits, _check_scenario, _same_snapshot, _snapshot

RECT = ([200.0], [300.0], [240.0], [320.0])  # around part of the fire and of the swarm's path
NONE = np.zeros((0, 5))
STAT4 = ("winner", "evaluations", "feasible", "removed")
STAT5 = STAT4 + ("appended",)


def _usage():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    return usage


# ---------------------------------------------------------------- CPU
@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_list_kernels_fit_their_launch():
    usage = _usage()
    for key in ("list_solve_kernel", "list_eval_kernel"):
        ks = [k for k in usage if key in k]
        assert len(ks) == 1, (key, ks)
        v = usage[ks[0]]
        assert v["LOCAL"] == 0 and v["STACK"] <= 128 and v["REG"] * 256 * 2 <= 65536, (key, v)
    counts = {"mads_kernel": 4, "scenario_solve_kernel": 2, "scenario_eval_kernel": 2, "region_solve_kernel": 1,
              "remove_covered_kernel": 1, "add_points_kernel": 1, "pack_planes_kernel": 1, "thresholds_kernel": 1,
              "ordered_kernel": 1}
    for key, n in counts.items():
        assert sum(key in k for k in usage) == n, key
    assert sum("horizon_start_kernel" in k or "horizon_commit_kernel" in k for k in usage) == 2


def test_option_constant(cov):
    assert cov.OPT_LIST_ORDER_HORIZON == cov._lib.OPT_LIST_ORDER_HORIZON == 11
    assert cov._lib.lib.cov_set_option(None, 11, 1) == cov._lib.COV_ERR_INVALID


def test_keyword_puts_the_option_back_when_the_call_raises(cov):
    opts, seen = {11: 0}, []

    def fail(*a, **k):
        seen.append(opts[11])
        raise cov.CoverageError(cov._lib.COV_ERR_STATE, "refused")

    stub = types.SimpleNamespace(get_option=lambda o: opts[o], set_option=lambda o, v: opts.__setitem__(o, v),
                                 N=5, _h=None, _horizon=fail, grid_info=lambda: {"nx": 2, "ny": 2})
    stub._check = fail
    E = cov.CoverageEngine
    calls = [lambda **k: E.run_horizon(stub, np.zeros(15), 2, **k),
             lambda **k: E.run_horizon_points(stub, np.zeros(15), [NONE], **k),
             lambda **k: E.run_horizon_ensemble(stub, np.zeros((2, 15)), 2, **k),
             lambda **k: E.run_horizon_points_ensemble(stub, np.zeros((2, 15)), [[NONE]], **k)]
    for prev in (0, 1):
        for call in calls:
            opts[11] = prev
            with pytest.raises(cov.CoverageError):
                call(list_order=True)
            assert seen[-1] == 1 and opts[11] == prev
            with pytest.raises(cov.CoverageError):
                call()
            assert seen[-1] == prev and opts[11] == prev  # without the keyword the option is left as it is


# ---------------------------------------------------------------- GPU: stores and the replay
def _rect(cov, pts):
    c = cov.CellFunctions.Cells()
    c.high_interest = RECT
    return c._reweight(np.asarray(pts, dtype=np.float64).reshape(-1, 5))


def _dyadic_rows(cov, fire_rows, first, T):
    """Rows first .. first + T - 1 of the fire table without the entries the rectangle would reweight (a cell keeps
    one weight across every schedule)."""
    rows = [np.asarray(fire_rows[first + t]).reshape(-1, 5) for t in range(T)]
    return [r[_rect(cov, r)[:, 3] == r[:, 3]] for r in rows]


def _swarm(cov, N, cx=250.0, cy=250.0):
    if N == 1:
        return np.array([cx, cy, 15.0 * T_HALF])
    if N == 64:  # 8 x 8 small discs, 14 m apart
        g = np.arange(8) * 14.0 - 49.0
        x, y = np.meshgrid(cx + g, cy + g, indexing="ij")
        return np.concatenate([x.ravel(), y.ravel(), np.full(64, 5.0 * T_HALF)])
    return cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, cx, cy)


def _static_store(cov, eng, case, fire_rows):
    """The case's list-order store and parameters on eng.  Returns (x0, kw)."""
    N = {"n1": 1, "n64": 64}.get(case, 5)
    x0 = _swarm(cov, N)
    kw = dict(S=8, spread=3.0, n_iter=40, granularity=1.0, seed=2**64 - 3, boxes=np.array([[220.0, 280.0, 230.0, 270.0]]),
              h_focus=15.0, h_max=30.0)
    T = 6
    init = np.concatenate([np.asarray(r).reshape(-1, 5) for r in fire_rows[:20]])
    if case in ("createpoi_s1", "createpoi_s32", "pending", "cons78", "gran0", "gran_half"):
        eng.set_points(_rect(cov, cov.AreaCoverageCalculation.createPOI(5.0, 5.0, 100.0, 100.0).data), 100, 100, 5.0, 5.0)
    else:
        eng.set_points(_rect(cov, init), 100, 100, 5.0, 5.0)
    if case == "createpoi_s1":
        kw.update(S=1, n_iter=100)
    elif case == "createpoi_s32":
        kw.update(S=32)
    elif case == "n64":
        kw.update(S=2, n_iter=3)
        T = 2
    elif case == "gran0":
        kw.update(granularity=0.0, n_iter=25)
    elif case == "gran_half":
        kw.update(granularity=0.5)
    elif case == "pending":  # a removal pending from an earlier cov_remove_covered: the list drops it lazily
        eng.remove_covered(_swarm(cov, 5, 300.0, 330.0))
    sep = 4.0 if case == "cons78" else 0.0
    eng.set_params(N, np.full(N, 30 * T_HALF), 1e5, prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF, sep_min=sep,
                   use_cons7=case == "cons78")
    assert eng.grid_info()["area_exact"] == 0
    return x0, T, kw, sep, case == "cons78"


def _setp(eng, N, sep, c7):
    def setp(r, prev):
        eng.set_params(N, r, 1e5, prev_xyR=prev, d_lim=10.0, tan_half_fov=T_HALF, sep_min=sep, use_cons7=c7)
    return setp


def _compare(X, obj, st, names, Xr, objr, str_):
    assert np.array_equal(_bits(X), _bits(Xr)), np.flatnonzero(np.any(X != Xr, axis=1))[:5]
    assert np.array_equal(_bits(obj), _bits(objr)), (obj, objr)
    got = np.stack([st[k] for k in names], axis=1)
    assert np.array_equal(got, str_[:, :len(names)]), (got, str_)


STATIC_CASES = ["createpoi_s1", "createpoi_s32", "cons78", "n1", "n64", "gran0", "gran_half", "pending"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", STATIC_CASES)
def test_static_horizon_bit_for_bit_against_single_calls(cov, engine, fire_rows, case):
    ref = cov.CoverageEngine(0)
    try:
        x0, T, kw, sep, c7 = _static_store(cov, engine, case, fire_rows)
        _static_store(cov, ref, case, fire_rows)
        N = x0.size // 3
        X, obj, st, ms = engine.run_horizon(x0, T, list_order=True, **kw)
        assert engine.get_option(cov.OPT_LIST_ORDER_HORIZON) == 0 and ms.shape == (T,) and np.all(ms > 0)
        Xr, objr, str_, _, _, _ = replay(cov.synth, ref, x0, T, kw["S"], kw["spread"], kw["n_iter"], kw["granularity"],
                                         kw["seed"], kw["boxes"], kw["h_focus"], kw["h_max"],
                                         np.full(N, 30 * T_HALF), _setp(ref, N, sep, c7), lambda t: 0)
        _compare(X, obj, st, STAT4, Xr, objr, str_)
        assert st["removed"].sum() > 0
        same_handles(cov, engine, ref, X, x0)
    finally:
        ref.close()


def _points_store(cov, eng, case, fire_rows):
    """The case's store, parameters and schedule on eng.  Returns (x0, appends, kw)."""
    N = 5
    x0 = _swarm(cov, N)
    kw = dict(S=8, spread=3.0, n_iter=60, granularity=1.0, seed=2**64 - 7, boxes=REF_BOXES, h_focus=15.0, h_max=30.0)
    init = np.concatenate([np.asarray(r).reshape(-1, 5) for r in fire_rows[:10]])
    c5 = [NONE] + [np.asarray(fire_rows[t + 9]).reshape(-1, 5) for t in range(2, 41)]
    if case.startswith("c5_s"):  # C5 with the rectangle: non-dyadic entries in the initial list and in the appends
        S = int(case[4:])
        kw.update(S=S, n_iter=100)
        T = 40 if S == 1 else 12
        eng.set_points(_rect(cov, init), 100, 100, 5.0, 5.0)
        appends = [_rect(cov, a) for a in c5[:T]]
    elif case == "mid":  # a dyadic store; the non-dyadic weight first appears at t = 4
        eng.set_points(init, 100, 100, 5.0, 5.0)
        appends = [a if t < 4 else _rect(cov, a) for t, a in enumerate(c5[:10], 1)]
    elif case == "refill":  # entries appended onto cells the first timestep emptied, and next to them
        c = np.arange(1, 101) * 5.0 - 2.5
        cx, cy = np.meshgrid(c, c, indexing="ij")
        d = np.min([np.hypot(cx - x0[i], cy - x0[N + i]) - x0[2 * N + i] for i in range(N)], axis=0)
        under = np.flatnonzero(d.T.ravel() < -2.0)
        fire = _rect(cov, init)
        eng.set_points(np.concatenate([fire[~np.isin(cell_of(fire), under)], _rect(cov, centres(under))]), 100, 100,
                       5.0, 5.0)
        appends = [NONE] * 10
        appends[2] = _rect(cov, centres(under[::3]))  # a cell keeps the one weight its position gives
        appends[5] = _rect(cov, centres(np.concatenate([under[::3], under[1::3]])))
        appends[8] = _rect(cov, centres(under[::2]))
        appends[4] = _rect(cov, c5[4])
    elif case == "no_list":  # a store without a list (createPOI's order fixed first), non-dyadic appends on cells
        eng.set_grid_full(100, 100, 5.0, 5.0)  # an earlier removal emptied
        away = _swarm(cov, N, 100.0, 400.0)
        eng.remove_covered(away)
        empty = np.flatnonzero(eng.grid_cells() == 0)
        nd = centres(empty)
        nd[:, 3] = (30 * T_HALF) ** 2 * math.pi
        appends = [NONE, nd[::2], NONE, nd[1::2], NONE, nd[::3]]
    elif case == "empty":
        eng.set_points(_rect(cov, init), 100, 100, 5.0, 5.0)
        appends = [NONE] * 8
    else:
        raise AssertionError(case)
    _params(eng, N)(np.full(N, 30 * T_HALF), x0)
    return x0, appends, kw


POINT_CASES = ["c5_s1", "c5_s148", "mid", "refill", "no_list", "empty"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", POINT_CASES)
def test_fire_list_bit_for_bit_against_single_calls(cov, engine, fire_rows, case):
    ref = cov.CoverageEngine(0)
    try:
        x0, appends, kw = _points_store(cov, engine, case, fire_rows)
        _points_store(cov, ref, case, fire_rows)
        if case != "mid":
            assert engine.grid_info()["area_exact"] == 0 or case == "no_list"
        T, N = len(appends), x0.size // 3
        X, obj, st, ms, last = engine.run_horizon_points(x0, appends, list_order=True, **kw)

        def add(t):
            if len(appends[t - 1]):
                ref.add_points(appends[t - 1])
            return len(appends[t - 1])

        Xr, objr, str_, _, lastr, _ = replay(cov.synth, ref, x0, T, kw["S"], kw["spread"], kw["n_iter"],
                                             kw["granularity"], kw["seed"], kw["boxes"], kw["h_focus"], kw["h_max"],
                                             np.full(N, 30 * T_HALF), _params(ref, N), add)
        _compare(X, obj, st, STAT5, Xr, objr, str_)
        assert np.array_equal(last, lastr)
        assert st["removed"].sum() > 0
        if case == "refill":
            ta = np.concatenate([np.full(len(a), t) for t, a in enumerate(appends, 1)])
            ci = cell_of(np.concatenate(appends))
            assert str_[0, 3] > 0 and (lastr[ci] >= ta).any()  # emptied at t = 1, refilled, removed again
        same_handles(cov, engine, ref, X, x0)
    finally:
        ref.close()


# ---------------------------------------------------------------- GPU: ensembles against the single calls
@pytest.mark.gpu
@pytest.mark.parametrize("E", [1, 5])
def test_static_ensemble_equals_cov_run_horizon(cov, engine, fire_rows, E):
    ref = cov.CoverageEngine(0)
    try:
        x0, T, kw, _, _ = _static_store(cov, engine, "createpoi_s32", fire_rows)
        kw.update(S=4)
        rng = np.random.default_rng(E)
        starts = np.repeat(x0[None], E, axis=0)
        starts[1:, :10] += np.rint(rng.uniform(-30, 30, size=(E - 1, 10)))
        C_, snap = _snapshot_static(cov, engine, 5)
        X, obj, st, ms, cells = engine.run_horizon_ensemble(starts, T, want_cells=True, list_order=True, **kw)
        _same_snapshot(engine, C_, snap)
        for e in range(E):
            _static_store(cov, ref, "createpoi_s32", fire_rows)
            Xr, objr, str_, _ = ref.run_horizon(starts[e], T, list_order=True,
                                                **dict(kw, seed=(kw["seed"] + e * T * kw["S"]) % 2**64))
            assert np.array_equal(_bits(X[e]), _bits(Xr)) and np.array_equal(_bits(obj[e]), _bits(objr)), e
            assert all(np.array_equal(st[k][e], str_[k]) for k in STAT4), e
            assert np.array_equal(cells[e], ref.grid_cells()), e
    finally:
        ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("E", [1, 5])
def test_points_ensemble_equals_cov_run_horizon_points(cov, engine, fire_rows, E):
    ref = cov.CoverageEngine(0)
    try:
        x0, appends, kw = _points_store(cov, engine, "c5_s148", fire_rows)
        kw.update(S=4, n_iter=60)
        T = 10
        schedules = [appends[:T], _dyadic_rows(cov, fire_rows, 12, T)]  # non-dyadic, dyadic
        list_of = np.array([0, 1, 1, 0, 1][:E], dtype=np.int64)
        rng = np.random.default_rng(E + 7)
        starts = np.repeat(x0[None], E, axis=0)
        starts[1:, :10] += np.rint(rng.uniform(-30, 30, size=(E - 1, 10)))
        C_, snap = _snapshot(cov, engine)
        X, obj, st, ms, cells, last = engine.run_horizon_points_ensemble(
            starts, schedules, list_of, want_cells=True, want_last_removed=True, list_order=True, **kw)
        _same_snapshot(engine, C_, snap)
        for e in range(E):
            _points_store(cov, ref, "c5_s148", fire_rows)
            Xr, objr, str_, _, lastr = ref.run_horizon_points(starts[e], schedules[list_of[e]], list_order=True,
                                                              **dict(kw, seed=(kw["seed"] + e * T * kw["S"]) % 2**64))
            _check_scenario(X, obj, st, cells, last, e, Xr, objr, str_, ref.grid_cells(), lastr)
        assert st["removed"].sum() > 0
    finally:
        ref.close()


# ---------------------------------------------------------------- GPU: run_simulation
def _sim_cells(cov, fire_rows):
    cells = cov.CellFunctions.Cells()
    cells.high_interest = RECT
    return cov.CellFunctions.initialise_POI(cells, "dynamic", fire_rows)


@pytest.mark.gpu
def test_run_simulation_list_order_equals_the_replay(cov, fire_rows):
    CF, FS, TC = cov.CellFunctions, cov.FullSimulation, cov.TDM_Constraints
    params = FS.SimulationParameters(N_iter=60, seed=29, environment_type="dynamic")
    N, steps, S = params.N, 12, 16
    start = _swarm(cov, N)
    r_max = params.h_max * T_HALF * np.ones(N)
    cells = _sim_cells(cov, fire_rows)
    ref = cov.CoverageEngine(0)
    try:
        with pytest.raises(cov.CoverageError) as err:  # without the keyword: refused as before
            FS.run_simulation(cells, start, TC.cons1, [], N, r_max.copy(), params, Nt_sim=steps, starts=S)
        assert err.value.code == cov._lib.COV_ERR_STATE
        inp, outp, runtimes, objs = FS.run_simulation(cells, start, TC.cons1, [], N, r_max, params, Nt_sim=steps,
                                                      starts=S, spread=2.0, list_order=True)
        init = _sim_cells(cov, fire_rows)
        data0 = init.points_of_interest.data.copy()
        sched = CF.update_POI_schedule(init, steps)
        init.close()
        ref.set_points(data0, 100, 100, 5.0, 5.0)
        assert ref.grid_info()["area_exact"] == 0

        def setp(r, prev):
            ref.set_params(N, r, 1e5, prev_xyR=prev, d_lim=params.d_lim, tan_half_fov=T_HALF)

        setp(params.h_max * T_HALF * np.ones(N), start)

        def add(t):
            if len(sched[t - 1]):
                ref.add_points(sched[t - 1])
            return len(sched[t - 1]), sched[t - 1]

        Xr, objr, _, r_end, _, hl = replay(cov.synth, ref, start, steps, S, 2.0, params.N_iter, 1.0, params.seed,
                                           FS._boxes(params), FS.H_FOCUS, params.h_max,
                                           params.h_max * T_HALF * np.ones(N), setp, add, hl=data0)
        assert np.array_equal(_bits(np.array(outp)), _bits(Xr)) and np.array_equal(_bits(objs), _bits(objr))
        assert np.array_equal(np.array(inp), np.concatenate([start[None], Xr[:-1]]))
        assert len(runtimes) == steps and np.array_equal(r_max, r_end)
        assert np.array_equal(cells.points_of_interest.data, hl)  # row for row
        eng = cells.resident().engine
        assert eng.get_option(cov.OPT_LIST_ORDER_HORIZON) == 0
        assert np.array_equal(eng.grid_cells(), ref.grid_cells()) and eng.grid_info() == ref.grid_info()
        same_handles(cov, eng, ref, Xr, start)
    finally:
        ref.close()
        cells.close()


@pytest.mark.gpu
def test_run_simulation_ensemble_list_order_equals_run_simulation(cov, fire_rows):
    FS, TC = cov.FullSimulation, cov.TDM_Constraints
    params = FS.SimulationParameters(N_iter=60, seed=31, environment_type="dynamic")
    N, steps, S = params.N, 8, 4
    base = _swarm(cov, N)
    swarms = [base, base + np.concatenate([np.full(N, 20.0), np.full(N, -15.0), np.zeros(N)]), base.copy()]
    r_max = params.h_max * T_HALF * np.ones(N)
    cells = _sim_cells(cov, fire_rows)
    try:
        data0 = cells.points_of_interest.data.copy()
        with pytest.raises(cov.CoverageError) as err:
            FS.run_simulation_ensemble(cells, swarms, TC.cons1, N, r_max, params, Nt_sim=steps, starts=S)
        assert err.value.code == cov._lib.COV_ERR_STATE
        out = FS.run_simulation_ensemble(cells, swarms, TC.cons1, N, r_max, params, Nt_sim=steps, starts=S,
                                         spread=2.0, list_order=True)
        assert np.array_equal(cells.points_of_interest.data, data0)
        for e, sw in enumerate(swarms):
            ce = _sim_cells(cov, fire_rows)
            try:
                pe = FS.SimulationParameters(N_iter=60, seed=params.seed + e * steps * S, environment_type="dynamic")
                ref = FS.run_simulation(ce, sw, TC.cons1, [], N, params.h_max * T_HALF * np.ones(N), pe, Nt_sim=steps,
                                        starts=S, spread=2.0, list_order=True)
            finally:
                ce.close()
            assert np.array_equal(np.array(out[e][0]), np.array(ref[0]))
            assert np.array_equal(_bits(np.array(out[e][1])), _bits(np.array(ref[1])))
            assert np.array_equal(_bits(out[e][3]), _bits(ref[3]))
    finally:
        cells.close()


# ---------------------------------------------------------------- GPU: the option itself
@pytest.mark.gpu
def test_option_round_trip(cov, engine):
    L = cov._lib
    assert engine.get_option(cov.OPT_LIST_ORDER_HORIZON) == 0
    for v in (1, 0, 1):
        engine.set_option(cov.OPT_LIST_ORDER_HORIZON, v)
        assert engine.get_option(cov.OPT_LIST_ORDER_HORIZON) == v
    for bad in (2, -1, 2**40):
        assert L.lib.cov_set_option(engine.handle, 11, bad) == L.COV_ERR_INVALID
        assert engine.get_option(cov.OPT_LIST_ORDER_HORIZON) == 1
    engine.set_option(cov.OPT_LIST_ORDER_HORIZON, 0)


@pytest.mark.gpu
def test_option_on_dyadic_stores_changes_nothing(cov, engine, fire_rows):
    ref = cov.CoverageEngine(0)
    try:
        N = 5
        x0 = _swarm(cov, N)
        init = np.concatenate([np.asarray(r).reshape(-1, 5) for r in fire_rows[:10]])
        sched = [NONE] + [np.asarray(fire_rows[t + 9]).reshape(-1, 5) for t in range(2, 7)]
        kw = dict(S=4, spread=3.0, n_iter=40, granularity=1.0, seed=99, boxes=REF_BOXES, h_focus=15.0, h_max=30.0)
        starts = np.stack([x0, x0 + np.concatenate([np.full(N, 10.0), np.zeros(2 * N)])])
        calls = [lambda e, lo: e.run_horizon(x0, 5, list_order=lo, **kw),
                 lambda e, lo: e.run_horizon_points(x0, sched, list_order=lo, **kw),
                 lambda e, lo: e.run_horizon_ensemble(starts, 5, want_cells=True, list_order=lo, **kw),
                 lambda e, lo: e.run_horizon_points_ensemble(starts, [sched], want_cells=True, want_last_removed=True,
                                                             list_order=lo, **kw)]
        for call in calls:
            outs = []
            for eng, lo in ((engine, True), (ref, False)):
                eng.set_points(init, 100, 100, 5.0, 5.0)
                _params(eng, N)(np.full(N, 30 * T_HALF), x0)
                n0 = eng.launch_count()
                out = call(eng, lo)
                outs.append((out, eng.launch_count() - n0))
            (a, na), (b, nb) = outs
            assert na == nb
            for i, (p, q) in enumerate(zip(a, b)):
                if isinstance(p, dict):
                    assert all(np.array_equal(p[k], q[k]) for k in p)
                elif i != 3:  # step_ms is a timing
                    assert np.array_equal(np.asarray(p).view(np.uint8), np.asarray(q).view(np.uint8)), i
            assert np.array_equal(engine.grid_cells(), ref.grid_cells())
    finally:
        ref.close()


@pytest.mark.gpu
def test_refusals_with_the_option_on(cov, engine, fire_rows):
    L = cov._lib
    N = 5
    x0 = _swarm(cov, N)
    engine.set_option(cov.OPT_LIST_ORDER_HORIZON, 1)
    try:
        # the automaton horizons: a fire store with a non-dyadic entry
        ff = cov.DynamicArea.ForestFire(engine, seed=3)
        nd = centres([0])
        nd[:, 3] = 0.1
        engine.add_points(nd)
        assert engine.grid_info()["area_exact"] == 0
        _params(engine, N)(np.full(N, 30 * T_HALF), x0)
        C_, snap = _snapshot(cov, engine)
        st0 = engine.fire_state()
        with pytest.raises(cov.CoverageError) as err:
            ff.run_horizon(x0, [1, 1], S=2, boxes=REF_BOXES)
        assert err.value.code == L.COV_ERR_STATE
        with pytest.raises(cov.CoverageError) as err:
            engine.run_horizon_fire_ensemble(np.stack([x0, x0]), [1, 1], (4.0, 4.7, 0.5), 3, 1, S=2, boxes=REF_BOXES)
        assert err.value.code == L.COV_ERR_STATE
        _same_snapshot(engine, C_, snap)
        assert np.array_equal(engine.fire_state(), st0)
        # more than 4 classes; mixed weights on one cell
        init = _rect(cov, np.concatenate([np.asarray(r).reshape(-1, 5) for r in fire_rows[:10]]))
        engine.set_points(init, 100, 100, 5.0, 5.0)
        _params(engine, N)(np.full(N, 30 * T_HALF), x0)
        C_, snap = _snapshot(cov, engine)
        free = np.flatnonzero(engine.grid_cells() == 0)[::-1]
        ws = [centres(free[k:k + 1]) for k in range(3)]
        for k, w in enumerate(ws):
            w[:, 3] = 0.1 * (k + 1)
        for call in (lambda s: engine.run_horizon_points(x0, s, S=2, boxes=REF_BOXES),
                     lambda s: engine.run_horizon_points_ensemble(np.stack([x0, x0]), [s], S=2, boxes=REF_BOXES)):
            with pytest.raises(cov.CoverageError) as err:
                call([NONE, ws[0], np.concatenate(ws[1:])])
            assert err.value.code == L.COV_ERR_LIMIT
            _same_snapshot(engine, C_, snap)
            other = centres(cell_of(init[:1]))
            other[:, 3] = 0.7
            with pytest.raises(cov.CoverageError) as err:
                call([NONE, other])
            assert err.value.code == L.COV_ERR_INVALID
            _same_snapshot(engine, C_, snap)
        # still usable, the option on
        X, obj, st, ms, last = engine.run_horizon_points(x0, [NONE, ws[0]], S=2, boxes=REF_BOXES)
        assert np.isfinite(obj).all() and list(st["appended"]) == [0, 1]
    finally:
        engine.set_option(cov.OPT_LIST_ORDER_HORIZON, 0)


# ---------------------------------------------------------------- GPU: several devices
@pytest.mark.gpu
def test_multi_device_equals_single_device(cov, engine, fire_rows):
    lib = cov._lib.lib
    x0, appends, kw = _points_store(cov, engine, "c5_s148", fire_rows)
    kw.update(S=2, n_iter=40)
    T = 8
    schedules = [appends[:T], _dyadic_rows(cov, fire_rows, 12, T)]
    E = 5
    list_of = np.array([0, 1, 0, 0, 1], dtype=np.int64)
    starts = np.repeat(x0[None], E, axis=0)
    starts[1:, :10] += np.rint(np.random.default_rng(3).uniform(-30, 30, size=(E - 1, 10)))
    X, obj, st, _, cells, last = engine.run_horizon_points_ensemble(starts, schedules, list_of, want_cells=True,
                                                                    want_last_removed=True, list_order=True, **kw)
    rows = [np.asarray(a, dtype=np.float64).reshape(-1, 5) for s in schedules for a in s]
    offsets = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    pts = np.ascontiguousarray(np.concatenate(rows))
    devs = (C.c_int * 2)(0, 1 if cov.device_count() >= 2 else 0)
    m = C.c_void_p()
    assert lib.cov_multi_create(devs, 2, C.byref(m)) == 0
    shards = []
    try:
        for k in range(2):
            sh = cov.CoverageEngine.__new__(cov.CoverageEngine)
            sh._h, sh._pinned, sh.N, sh.device, sh.param_owner = C.c_void_p(lib.cov_multi_handle(m, k)), [], None, devs[k], None
            shards.append(sh)
            _points_store(cov, sh, "c5_s148", fire_rows)
            sh.set_option(cov.OPT_LIST_ORDER_HORIZON, 1)
        n = starts.shape[1]
        Xm, om = np.empty((E, T, n)), np.empty((E, T))
        sm, cm, lm = np.empty((E, T, 5), dtype=np.int64), np.empty_like(cells), np.empty_like(last)
        B = kw["boxes"]
        assert lib.cov_multi_run_horizon_points_ensemble(m, starts.ctypes.data, E, T, kw["S"], kw["spread"],
                                                         kw["n_iter"], kw["granularity"], kw["seed"], B.ctypes.data,
                                                         len(B), kw["h_focus"], kw["h_max"], pts.ctypes.data,
                                                         offsets.ctypes.data, len(schedules), list_of.ctypes.data,
                                                         Xm.ctypes.data, om.ctypes.data, sm.ctypes.data,
                                                         cm.ctypes.data, lm.ctypes.data) == 0, \
            lib.cov_multi_last_error(m)
        assert np.array_equal(_bits(Xm), _bits(X)) and np.array_equal(_bits(om), _bits(obj))
        assert np.array_equal(sm, np.stack([st[k] for k in STAT5], axis=2))
        assert np.array_equal(cm, cells) and np.array_equal(lm, last)
    finally:
        for sh in shards:
            sh._h = None
        lib.cov_multi_destroy(m)
