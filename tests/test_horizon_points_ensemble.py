"""cov_run_horizon_points_ensemble: E independent dynamic receding horizons over the reference's fire list in one call,
each with its own starting swarm and one of L fire schedules, on private copies of the handle's store and parameters.

CPU: what nvcc built for the append and removal kernels, which gained a scenario dimension, and the solver inventory
around them; the refusals that need no device; the engine wrapper's shape checks.  GPU: every scenario bit for bit
against cov_run_horizon_points on a twin handle holding the same store and parameters, with seed + e * T * S and
schedule list_of[e] (X, objectives, all five stats columns, the cells it leaves, last_removed); the handle is unchanged,
refusals included; run_simulation_ensemble(environment_type="dynamic") against run_simulation; the multi-device call
against the single-device one.
"""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from test_horizon_dynamic import cell_of, centres, same_handles

T_HALF = math.tan((100 / 180 * math.pi) / 2)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "maximumareacoverageoptimization.jl_b200", "libcoverage_cuda.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
REF_BOXES = np.array([[2500.0, 3500.0, 1000.0, 2000.0]])  # SimulationParameters' rectangle: outside the 500 m domain
STAT_NAMES = ("winner", "evaluations", "feasible", "removed", "appended")
NONE = np.zeros((0, 5))
N = 5


# ---------------------------------------------------------------- CPU
@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_store_kernels_fit_their_launch():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    for key in ("add_points_kernel", "remove_covered_kernel"):
        ks = [k for k in usage if key in k]
        assert len(ks) == 1, (key, ks)  # the scenario dimension is a run-time argument, not an instantiation
        v = usage[ks[0]]
        assert v["LOCAL"] == 0 and v["STACK"] == 0 and v["REG"] * 256 <= 65536, (key, v)  # 256-thread CTAs
    # the solver around them is unchanged
    assert sum("mads_kernel" in k for k in usage) == 4
    assert sum("horizon_start_kernel" in k or "horizon_commit_kernel" in k for k in usage) == 2
    assert sum("scenario_solve_kernel" in k for k in usage) == 2 and sum("scenario_eval_kernel" in k for k in usage) == 2


def test_refusals_without_a_device(cov):
    L = cov._lib
    lib = L.lib
    x = np.zeros(3 * N)
    X = np.empty(3 * N)
    off = np.zeros(2, dtype=np.int64)
    lo = np.zeros(1, dtype=np.int64)
    assert lib.cov_run_horizon_points_ensemble(None, x.ctypes.data, 1, 1, 1, 3.0, 10, 1.0, 0, None, 0, 15.0, 30.0,
                                               None, off.ctypes.data, 1, lo.ctypes.data, X.ctypes.data, None, None,
                                               None, None, None) == L.COV_ERR_INVALID
    assert lib.cov_multi_run_horizon_points_ensemble(None, x.ctypes.data, 1, 1, 1, 3.0, 10, 1.0, 0, None, 0, 15.0,
                                                     30.0, None, off.ctypes.data, 1, lo.ctypes.data, X.ctypes.data,
                                                     None, None, None, None) == L.COV_ERR_INVALID


def test_engine_shape_errors(cov):
    eng = cov.CoverageEngine.__new__(cov.CoverageEngine)  # no device: every check comes before the library call
    eng._h, eng.N = None, N
    xs = np.zeros((2, 3 * N))
    two = [[NONE, NONE], [NONE, NONE]]
    for bad in (dict(x_starts=np.zeros((2, 14))), dict(x_starts=np.zeros((2, 2, 3 * N))), dict(schedules=[]),
                dict(schedules=[[NONE, NONE], [NONE]]), dict(list_of=[0]), dict(list_of=[0, 0, 0]),
                dict(list_of=[0, 2]), dict(list_of=[-1, 0]), dict(list_of=[[0, 1]])):
        kw = dict(x_starts=xs, schedules=two, list_of=[1, 0])
        kw.update(bad)
        with pytest.raises(ValueError):
            eng.run_horizon_points_ensemble(**kw)
    eng.N = None
    with pytest.raises(ValueError):  # no set_params yet
        eng.run_horizon_points_ensemble(xs, two)


# ---------------------------------------------------------------- GPU: against cov_run_horizon_points on a twin handle
def _params(eng, prev):
    eng.set_params(N, np.full(N, 30 * T_HALF), 1e5, prev_xyR=prev, d_lim=10.0, tan_half_fov=T_HALF)


def _c5(fire_rows, T, shift=0):
    """update_POI's schedule of BASELINE C5 (rows 1..10 in the store, row t + 10 appended at timestep t >= 2), its
    rows `shift` rows further on."""
    return [NONE] + [np.asarray(fire_rows[t + 9 + shift]).reshape(-1, 5) for t in range(2, T + 1)]


def _under(x, nx=100, d=5.0, margin=-2.0):
    """The cells whose centres lie inside the swarm x's discs by more than -margin metres."""
    c = np.arange(1, nx + 1) * d - d / 2
    cx, cy = np.meshgrid(c, c, indexing="ij")
    dist = np.min([np.hypot(cx - x[i], cy - x[N + i]) - x[2 * N + i] for i in range(N)], axis=0)
    return np.flatnonzero(dist.T.ravel() < margin)


def _prep(cov, eng, case, fire_rows):
    """The case's store and parameters on eng.  Returns (x_starts (E, 3N), schedules, list_of (E,), kw)."""
    rng = np.random.default_rng(sum(map(ord, case)))
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    E, S, T, n_iter, move = 3, 4, 10, 60, 40
    init = np.concatenate([np.asarray(r).reshape(-1, 5) for r in fire_rows[:10]])
    free = np.setdiff1d(np.arange(10000), cell_of(np.concatenate(fire_rows)))  # no fire entry ever lands there
    starts, list_of = None, None
    if case == "c5_e1":
        E, S, T, n_iter = 1, 1, 40, 100
        eng.set_points(init, 100, 100, 5.0, 5.0)
        schedules = [_c5(fire_rows, T)]
    elif case in ("three_schedules", "force_exact"):  # C5, C5 three timesteps late, nothing
        T = 12
        eng.set_points(init, 100, 100, 5.0, 5.0)
        c5 = _c5(fire_rows, T)
        schedules = [c5, [NONE] * 3 + c5[:T - 3], [NONE] * T]
        starts, list_of = np.repeat(x0[None], 3, axis=0), [0, 1, 2]
        if case == "force_exact":
            eng.set_option(cov.OPT_FORCE_EXACT, 1)
            E, starts, list_of = 4, None, [2, 0, 1, 0]
    elif case == "new_weight":  # 12.5 first appears at t = 4 in schedule 1 only, 6.25 at t = 3 in schedule 2
        E, T = 4, 8
        eng.set_points(init, 100, 100, 5.0, 5.0)
        c = free[np.hypot((free % 100 + 0.5) * 5 - 250, (free // 100 + 0.5) * 5 - 250) < 70]
        a, b = centres(c[0::6][:8]), centres(c[3::6][:8])
        a[:, 3], b[:, 3] = 12.5, 6.25
        s1, s2 = _c5(fire_rows, T), _c5(fire_rows, T)
        s1[3] = np.concatenate([s1[3], a])
        s2[2] = np.concatenate([b[:4], s2[2]])
        s2[5] = np.concatenate([s2[5], b[4:], b[4:]])
        schedules = [_c5(fire_rows, T), s1, s2]
        list_of = [2, 1, 0, 2]
    elif case == "dups_pow2":  # duplicates within a timestep on a full grid, onto cells scenario 0 emptied at t = 1
        E, T = 4, 8
        eng.set_grid_full(100, 100, 5.0, 5.0)
        u0 = _under(x0)
        ring = np.setdiff1d(_under(x0, margin=8.0), _under(x0, margin=1.0))
        far = np.arange(0, 30)  # row j = 1, x <= 150 m: no swarm reaches it
        a, b = [NONE] * T, [NONE] * T
        a[1] = centres(np.repeat(np.concatenate([far, ring[::3]]), 3))                # 1 -> 4
        a[3] = centres(np.concatenate([np.repeat(np.concatenate([far, ring[::3]]), 4), ring[1::5]]))  # 4 -> 8
        b[2] = centres(np.repeat(u0[::2], 5))                          # 0 -> 5 in scenario 0, 1 -> 6 elsewhere
        b[5] = centres(np.repeat(np.concatenate([u0[1::4], ring[::7]]), 2))
        schedules = [a, b]
        list_of = [1, 0, 1, 0]
        starts = np.repeat(x0[None], E, axis=0)
        starts[1:, :2 * N] += np.rint(rng.uniform(-40, 40, size=(E - 1, 2 * N)))
    elif case == "e148_s1":
        E, S, T, n_iter = 148, 1, 5, 40
        eng.set_points(init, 100, 100, 5.0, 5.0)
        schedules = [_c5(fire_rows, T)]
    elif case == "e300_s2_l8":  # more scenarios than one wave of persistent CTAs
        E, S, T, n_iter = 300, 2, 4, 30
        eng.set_points(init, 100, 100, 5.0, 5.0)
        schedules = [_c5(fire_rows, T, shift=3 * l) for l in range(8)]
        list_of = rng.integers(0, 8, size=E)
    elif case == "odd_lattice":  # 37 x 29 cells: scenario e's store starts mid-word for odd e
        E, T, move = 5, 8, 15
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 92.0, 72.0)
        nc = 37 * 29
        eng.set_points(centres(rng.choice(nc, 300), nx=37), 37, 29, 5.0, 5.0)
        schedules = []
        for _ in range(2):
            s = [NONE] + [centres(rng.choice(nc, int(rng.integers(20, 80))), nx=37) for _ in range(T - 1)]
            s[2] = np.concatenate([s[2], centres(np.repeat(rng.choice(nc, 10), 3), nx=37)])
            schedules.append(s)
        list_of = [0, 1, 1, 0, 1]
    else:
        raise AssertionError(case)
    if starts is None:  # distinct starts, scenario 0 unmoved
        starts = np.repeat(x0[None], E, axis=0)
        starts[1:, :2 * N] += np.rint(rng.uniform(-move, move, size=(E - 1, 2 * N)))
    list_of = np.zeros(E, dtype=np.int64) if list_of is None else np.asarray(list_of, dtype=np.int64)
    _params(eng, x0)
    kw = dict(S=S, spread=3.0, n_iter=n_iter, granularity=1.0, seed=2**64 - 5, boxes=REF_BOXES, h_focus=15.0,
              h_max=30.0)
    return starts, schedules, list_of, kw


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _snapshot(cov, eng, seed=11):
    C_ = cov.synth.random_candidates(1000, N, seed=seed)
    return C_, (eng.grid_cells(), eng.grid_info(), eng.class_weights(), eng.eval_batch(C_))


def _same_snapshot(eng, C_, snap):
    cells, info, cw, ev = snap
    assert np.array_equal(eng.grid_cells(), cells)
    assert eng.grid_info() == info and eng.class_weights() == cw
    now = eng.eval_batch(C_)
    for k in ev:
        assert np.array_equal(np.asarray(now[k]).view(np.uint8), np.asarray(ev[k]).view(np.uint8)), k


def _check_scenario(X, obj, st, cells, last, e, Xr, objr, str_, cells_r, last_r):
    assert np.array_equal(_bits(X[e]), _bits(Xr)), (e, np.flatnonzero(np.any(X[e] != Xr, axis=1))[:5])
    assert np.array_equal(_bits(obj[e]), _bits(objr)), (e, obj[e], objr)
    for k in STAT_NAMES:
        assert np.array_equal(st[k][e], str_[k]), (e, k, st[k][e], str_[k])
    assert np.array_equal(cells[e], cells_r), e
    assert np.array_equal(last[e], last_r), e


CASES = ["c5_e1", "three_schedules", "new_weight", "dups_pow2", "e148_s1", "e300_s2_l8", "odd_lattice", "force_exact"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_every_scenario_equals_cov_run_horizon_points(cov, engine, fire_rows, case):
    ref = cov.CoverageEngine(0)
    try:
        starts, schedules, list_of, kw = _prep(cov, engine, case, fire_rows)
        E, T, S, seed = starts.shape[0], len(schedules[0]), kw["S"], kw["seed"]
        C_, snap = _snapshot(cov, engine)
        launches = engine.launch_count()
        X, obj, st, ms, cells, last = engine.run_horizon_points_ensemble(starts, schedules, list_of, want_cells=True,
                                                                         want_last_removed=True, **kw)
        if E > 1:  # one launch per step for all E, an append only where some scenario's schedule has rows
            appends = sum(any(len(schedules[l][t]) for l in set(list_of.tolist())) for t in range(T))
            assert engine.launch_count() - launches == 1 + appends + 6 * T
        ncell = engine.grid_info()["nx"] * engine.grid_info()["ny"]
        assert X.shape == (E, T, 3 * N) and obj.shape == (E, T) and ms.shape == (T,) and np.all(ms > 0)
        assert cells.shape == last.shape == (E, ncell) and last.dtype == np.int32
        _same_snapshot(engine, C_, snap)  # the handle is unchanged
        for e in range(E):
            _prep(cov, ref, case, fire_rows)
            Xr, objr, str_, _, lastr = ref.run_horizon_points(starts[e], schedules[list_of[e]],
                                                              **dict(kw, seed=(seed + e * T * S) % 2**64))
            _check_scenario(X, obj, st, cells, last, e, Xr, objr, str_, ref.grid_cells(), lastr)
            assert np.array_equal(st["appended"][e], [len(a) for a in schedules[list_of[e]]])
        assert st["removed"].sum() > 0
        if case == "c5_e1":
            assert st["appended"].sum() == 3474
        if case == "three_schedules":
            app = st["appended"]
            assert not np.array_equal(app[0], app[1]) and app[1].sum() > 0 and not app[2].any()
            third = cov.CoverageEngine(0)  # the empty schedule is cov_run_horizon_ensemble's scenario
            try:
                _prep(cov, third, case, fire_rows)
                Xs, objs, sts, _, cs = third.run_horizon_ensemble(starts, T, want_cells=True, **kw)
                assert np.array_equal(_bits(Xs[2]), _bits(X[2])) and np.array_equal(_bits(objs[2]), _bits(obj[2]))
                assert all(np.array_equal(sts[k][2], st[k][2]) for k in sts) and np.array_equal(cs[2], cells[2])
            finally:
                third.close()
        if case == "new_weight":  # the ensemble numbers 12.5 before 6.25; scenario 0's single call only has 6.25
            _prep(cov, ref, case, fire_rows)
            ref.run_horizon_points(starts[0], schedules[2], **dict(kw, n_iter=2))
            assert ref.class_weights()[:2] == [25.0, 6.25]
        if case == "dups_pow2":  # multiplicities 1 -> 4 -> 8 where no swarm removes them
            assert np.all(cells[1][:30] == 8) and np.all(cells[0][:30] == 1) and last[0].any()
        if case == "e300_s2_l8":  # a scenario does not depend on the ensemble around it
            for e in (0, 151, 299):
                out = engine.run_horizon_points_ensemble(starts[e:e + 1], schedules, list_of[e:e + 1],
                                                         want_cells=True, want_last_removed=True,
                                                         **dict(kw, seed=(seed + e * T * S) % 2**64))
                Xe, oe, se, _, ce, le = out
                _check_scenario(X, obj, st, cells, last, e, Xe[0], oe[0], {k: v[0] for k, v in se.items()}, ce[0],
                                le[0])
    finally:
        ref.close()


@pytest.mark.gpu
def test_handle_unchanged_with_pending_removals(cov, engine, fire_rows):
    twin = cov.CoverageEngine(0)
    try:
        starts, schedules, list_of, kw = _prep(cov, engine, "three_schedules", fire_rows)
        _prep(cov, twin, "three_schedules", fire_rows)
        first = np.concatenate([np.asarray(r).reshape(-1, 5) for r in fire_rows[:1]])
        hole = np.array([first[0, 0], first[0, 1], 12.0])
        for eng in (engine, twin):  # removals pending in the handle's ordered list
            assert eng.remove_covered(hole) > 0
        C_, snap = _snapshot(cov, engine)
        X, obj, st, ms = engine.run_horizon_points_ensemble(starts, schedules, list_of, **kw)
        assert st["appended"].sum() > 0 and st["removed"].sum() > 0
        _same_snapshot(engine, C_, snap)
        same_handles(cov, engine, twin, X[0], starts[0])  # through a non-dyadic entry: the ordered lists agree
    finally:
        twin.close()


@pytest.mark.gpu
def test_refusals_leave_the_handle_unchanged(cov, engine, fire_rows):
    L_ = cov._lib
    lib, h = L_.lib, engine.handle
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    xs = np.stack([x0, x0])
    Xo = np.empty((2, 4, 3 * N))
    init = np.concatenate([np.asarray(r).reshape(-1, 5) for r in fire_rows[:10]])
    free = np.setdiff1d(np.arange(10000), cell_of(init))[::-1]  # from the far corner

    def call(scheds=((NONE,) * 4, (NONE,) * 4), list_of=(0, 1), E=2, T=4, S=2, L=None, offsets=None, Xo_=Xo):
        rows = [np.asarray(a, dtype=np.float64).reshape(-1, 5) for s in scheds for a in s]
        off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64) if offsets is None else offsets
        P = np.ascontiguousarray(np.concatenate(rows)) if rows else NONE
        lo = None if list_of is None else np.ascontiguousarray(list_of, dtype=np.int64)
        return lib.cov_run_horizon_points_ensemble(h, xs.ctypes.data, E, T, S, 3.0, 5, 1.0, 0, REF_BOXES.ctypes.data,
                                                   1, 15.0, 30.0, P.ctypes.data if len(P) else None, off.ctypes.data,
                                                   len(scheds) if L is None else L,
                                                   None if lo is None else lo.ctypes.data,
                                                   None if Xo_ is None else Xo_.ctypes.data, None, None, None, None,
                                                   None)

    assert call() == L_.COV_ERR_STATE  # no grid
    engine.set_points(init, 100, 100, 5.0, 5.0)
    engine.set_params(N, np.full(N, 30 * T_HALF))
    assert call() == L_.COV_ERR_STATE  # cons3 off
    _params(engine, x0)
    C_, snap = _snapshot(cov, engine)
    row = centres(free[:1])
    bad_off = np.array([0, 0, 1, 1, 1, 0, 1, 1, 1], dtype=np.int64)  # falls where schedule 1 starts
    for bad in (dict(list_of=None), dict(list_of=(0, 2)), dict(list_of=(-1, 0)), dict(L=0), dict(L=-1),
                dict(scheds=((NONE, row, NONE, NONE), (NONE,) * 4), offsets=bad_off),
                dict(offsets=np.array([1, 1, 1, 1, 1, 1, 1, 1, 1], dtype=np.int64)),
                dict(E=0), dict(E=-1), dict(E=2**30, S=2), dict(S=0), dict(Xo_=None)):
        assert call(**bad) == L_.COV_ERR_INVALID, bad
        _same_snapshot(engine, C_, snap)
    assert call(T=0, offsets=np.zeros(1, dtype=np.int64), list_of=None) == L_.COV_OK  # nothing to do
    _same_snapshot(engine, C_, snap)
    # two weights on one cell across two schedules (each schedule alone has one)
    other = row.copy()
    other[:, 3] = 12.5
    assert call(scheds=((NONE, row, NONE, NONE), (NONE, NONE, other, NONE))) == L_.COV_ERR_INVALID
    _same_snapshot(engine, C_, snap)
    # more than 4 classes over the union of the schedules (each schedule alone brings 3)
    ws = [centres(free[1 + k:2 + k]) for k in range(4)]
    for k, w in enumerate(ws):
        w[:, 3] = 25.0 / 2 ** (k + 1)
    assert call(scheds=((NONE, ws[0], ws[1], NONE), (NONE, NONE, ws[2], ws[3]))) == L_.COV_ERR_LIMIT
    _same_snapshot(engine, C_, snap)
    # a schedule no scenario uses, whose weight would make the store's area depend on the list order
    nd = row.copy()
    nd[:, 3] = 0.1
    assert call(scheds=((NONE,) * 4, (NONE, NONE, nd, NONE)), list_of=(0, 0)) == L_.COV_ERR_STATE
    _same_snapshot(engine, C_, snap)
    # a cell past 255 in one schedule only; the bound is the largest schedule's, not their sum
    cell = centres(free[10:11])
    engine.add_points(np.repeat(cell, 200, axis=0))
    _params(engine, x0)
    C_, snap = _snapshot(cov, engine)
    assert call(scheds=((NONE, np.repeat(cell, 30, axis=0), NONE, NONE),
                        (NONE, NONE, np.repeat(cell, 60, axis=0), NONE))) == L_.COV_ERR_LIMIT
    _same_snapshot(engine, C_, snap)
    assert call(scheds=((NONE, np.repeat(cell, 50, axis=0), NONE, NONE),
                        (NONE, np.repeat(cell, 20, axis=0), np.repeat(cell, 30, axis=0), NONE))) == L_.COV_OK
    _same_snapshot(engine, C_, snap)


# ---------------------------------------------------------------- GPU: run_simulation_ensemble, dynamic
@pytest.mark.gpu
def test_run_simulation_ensemble_dynamic_equals_run_simulation(cov, fire_rows):
    CF, FS, TC = cov.CellFunctions, cov.FullSimulation, cov.TDM_Constraints
    params = FS.SimulationParameters(N_iter=60, seed=23, environment_type="dynamic")
    steps, S = 8, 4
    base = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    swarms = [base, base + np.concatenate([np.full(N, 20.0), np.full(N, -15.0), np.zeros(N)]), base.copy()]
    cells = CF.initialise_POI(CF.Cells(), "dynamic", fire_rows)
    try:
        r_max = params.h_max * T_HALF * np.ones(N)
        r_keep = r_max.copy()
        data0, n_xy = cells.points_of_interest.data.copy(), len(cells.fire_point_xy_ccordinates)
        out = FS.run_simulation_ensemble(cells, swarms, TC.cons1, N, r_max, params, Nt_sim=steps, starts=S, spread=2.0)
        assert len(out) == len(swarms)
        assert np.array_equal(r_max, r_keep)  # the caller's r_max
        assert np.array_equal(cells.points_of_interest.data, data0) and len(cells.fire_point_xy_ccordinates) == n_xy
        assert cells.resident().engine.grid_info()["n_entries"] == len(data0)  # and the resident store
        for e, sw in enumerate(swarms):
            ce = CF.initialise_POI(CF.Cells(), "dynamic", fire_rows)
            try:
                pe = FS.SimulationParameters(N_iter=60, seed=params.seed + e * steps * S, environment_type="dynamic")
                ref = FS.run_simulation(ce, sw, TC.cons1, [], N, params.h_max * T_HALF * np.ones(N), pe, Nt_sim=steps,
                                        starts=S, spread=2.0)
            finally:
                ce.close()
            inp, outp, rt, objs = out[e]
            assert np.array_equal(np.array(inp), np.array(ref[0])) and np.array_equal(np.array(outp), np.array(ref[1]))
            assert np.array_equal(_bits(objs), _bits(ref[3]))
            assert len(rt) == steps and all(r > 0 for r in rt)
        assert not np.array_equal(np.array(out[0][1]), np.array(out[2][1]))  # same start, other seed
        # a reweighted schedule whose area would depend on the list order (a rectangle around an appended entry on a
        # cell the store does not hold): refused, as run_simulation refuses it
        pts = np.concatenate(CF.update_POI_schedule(cells, steps))
        x, y = pts[~np.isin(cell_of(pts), cell_of(data0))][0, :2]
        single = CF.initialise_POI(CF.Cells(), "dynamic", fire_rows)
        try:
            for c in (cells, single):
                c.high_interest = ([x - 1], [x + 1], [y - 1], [y + 1])
            with pytest.raises(cov.CoverageError) as err:
                FS.run_simulation_ensemble(cells, swarms, TC.cons1, N, r_max, params, Nt_sim=steps, starts=S)
            assert err.value.code == cov._lib.COV_ERR_STATE
            assert np.array_equal(cells.points_of_interest.data, data0)
            with pytest.raises(cov.CoverageError) as err:
                FS.run_simulation(single, swarms[0], TC.cons1, [], N, r_max.copy(), params, Nt_sim=steps, starts=S)
            assert err.value.code == cov._lib.COV_ERR_STATE
        finally:
            single.close()
    finally:
        cells.close()


# ---------------------------------------------------------------- GPU: several devices
@pytest.mark.gpu
def test_multi_device_equals_single_device(cov, engine, fire_rows):
    lib = cov._lib.lib
    starts, schedules, list_of, kw = _prep(cov, engine, "new_weight", fire_rows)
    starts = np.concatenate([starts, starts[::-1][:3]])  # 7 scenarios: uneven shards
    list_of = np.concatenate([list_of, list_of[::-1][:3]])
    E, n, T = starts.shape[0], starts.shape[1], len(schedules[0])
    X, obj, st, _, cells, last = engine.run_horizon_points_ensemble(starts, schedules, list_of, want_cells=True,
                                                                    want_last_removed=True, **kw)
    rows = [np.asarray(a, dtype=np.float64).reshape(-1, 5) for s in schedules for a in s]
    offsets = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    pts = np.ascontiguousarray(np.concatenate(rows))
    devs = (C.c_int * 2)(0, 0)
    m = C.c_void_p()
    assert lib.cov_multi_create(devs, 2, C.byref(m)) == 0
    shards = []
    try:
        for k in range(2):
            sh = cov.CoverageEngine.__new__(cov.CoverageEngine)
            sh._h, sh._pinned, sh.N, sh.device, sh.param_owner = C.c_void_p(lib.cov_multi_handle(m, k)), [], None, 0, None
            shards.append(sh)
            _prep(cov, sh, "new_weight", fire_rows)
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
        assert np.array_equal(sm, np.stack([st[k] for k in STAT_NAMES], axis=2))
        assert np.array_equal(cm, cells) and np.array_equal(lm, last)
    finally:
        for sh in shards:
            sh._h = None
        lib.cov_multi_destroy(m)
