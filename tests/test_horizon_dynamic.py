"""cov_run_horizon_points / cov_run_horizon_fire: the dynamic receding horizon (update_POI's fire list or the device
automaton appending before every timestep's rmvCoveredPOI) on the device in one call.

CPU: the update_POI schedule builder; ForestFire.run_horizon's step bookkeeping; what nvcc built for the extended
removal kernel.  GPU: every horizon bit for bit against the same horizon replayed from single calls (cov_add_points
or cov_fire_step(append=1), cov_remove_covered, the rule in NumPy, cov_set_params, cov_mads_solve_batch on the model's
starts, a host argmin, cov_eval_batch), both handles alike afterwards (the ordered list included, through one
non-dyadic entry added on both); the error classes, each leaving the handle as it was; run_simulation(starts=S) with
the dynamic environment.
"""
import math
import os
import re
import subprocess
import types

import numpy as np
import pytest

from test_horizon import CUOBJDUMP, LIB, REF_BOXES, T_HALF, libm_b, model_starts, rule, table_b

M32 = 0xFFFFFFFF
WIND = (4.0, math.radians(270.0), 0.5)  # ForestFire's defaults: wind speed, direction, prob_spread


def centres(ci, nx=100, d=5.0):
    """Reference 5-tuples (weight d*d) on the 0-based cells ci of an nx-wide lattice."""
    ci = np.asarray(ci)
    i, j = ci % nx + 1, ci // nx + 1
    return np.stack([i * d - d / 2, j * d - d / 2, np.full(ci.size, d * d), np.full(ci.size, d * d),
                     np.zeros(ci.size)], axis=1)


def cell_of(pts, nx=100, d=5.0):
    return (np.rint((pts[:, 0] + d / 2) / d).astype(np.int64) - 1) + nx * (np.rint((pts[:, 1] + d / 2) / d).astype(np.int64) - 1)


# ---------------------------------------------------------------- CPU
def test_update_poi_schedule(cov, fire_rows):
    CF = cov.CellFunctions
    cells = CF.initialise_POI(CF.Cells(), "dynamic", fire_rows)
    sched = CF.update_POI_schedule(cells, 5)
    assert len(sched) == 5 and sched[0].shape == (0, 5)
    for t in range(2, 6):  # row t + 10 (1-based) of the table
        assert np.array_equal(sched[t - 1], np.asarray(fire_rows[t + 9]).reshape(-1, 5))
    # the table runs out: nothing more; update_POI's own appends are the same rows
    tail = CF.update_POI_schedule(cells, len(fire_rows))
    assert all(len(a) == 0 for a in tail[len(fire_rows) - 10:]) and len(tail[len(fire_rows) - 11]) > 0
    # reweighted as update_POI reweights (a rectangle around the first appended row's first point)
    x, y = sched[1][0, :2]
    cells.high_interest = ([x - 1], [x + 1], [y - 1], [y + 1])
    w = CF.update_POI_schedule(cells, 2)[1]
    inside = (np.abs(sched[1][:, 0] - x) < 1) & (np.abs(sched[1][:, 1] - y) < 1)
    assert np.all(w[inside, 3] == (cells.h_max * cells.tan_half_fov) ** 2 * math.pi)
    assert np.array_equal(w[~inside], sched[1][~inside]) and np.array_equal(w[:, :3], sched[1][:, :3])
    with pytest.raises(ValueError):
        CF.update_POI_schedule(CF.Cells(), 3)


def test_forest_fire_run_horizon_continues_the_step_stream(cov):
    calls = []
    eng = types.SimpleNamespace(
        fire_init=lambda *a, **k: None,
        run_horizon_fire=lambda *a, **k: calls.append(("horizon", a, k)) or "out",
        fire_step=lambda *a, **k: calls.append(("step", a, k)) or 0)
    ff = cov.DynamicArea.ForestFire(eng, seed=9)
    ff.step()
    ff.step()
    assert ff.run_horizon(np.zeros(15), [2, 0, 3], S=4) == "out"
    _, a, k = calls[-1]
    assert list(a[1]) == [2, 0, 3] and a[2:7] == (ff.wind_speed, ff.wind_direction, ff.prob_spread, 9, 3)
    assert k == {"S": 4} and ff.t == 7
    ff.step()
    assert calls[-1][1][4] == 8  # the next step() continues at 2 + 5 + 1
    ff.run_horizon(np.zeros(15), [0, 0])
    assert calls[-1][1][6] == 9 and ff.t == 8


@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_removal_kernel_fits_its_launch():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    rm = {k: v for k, v in usage.items() if "remove_covered_kernel" in k}
    assert len(rm) == 1, sorted(rm)
    for k, v in rm.items():
        assert v["LOCAL"] == 0 and v["STACK"] == 0, (k, v)
        assert v["REG"] * 256 <= 65536, (k, v)  # 256-thread CTAs
    assert sum("horizon_start_kernel" in k or "horizon_commit_kernel" in k for k in usage) == 2


# ---------------------------------------------------------------- GPU: the replay from single calls
def replay(synth, eng, x_start, T, S, spread, n_iter, g, seed, boxes, h_focus, h_max, r_max, setp, append, hl=None):
    """The horizon from single calls; append(t) = the timestep's appends (returns how many entries).  hl: a host
    list (P x 5) kept as update_POI and rmvCoveredPOI keep it.  Returns X, obj, stats (T x 5), r_max, last_removed,
    hl."""
    gi = eng.grid_info()
    cur, r_max = x_start.copy(), r_max.copy()
    last = np.zeros(gi["nx"] * gi["ny"], dtype=np.int32)
    X, obj, st = [], [], []
    for t in range(1, T + 1):
        appended = append(t)
        if hl is not None:
            hl = np.concatenate([hl, *appended[1:]])
            appended = appended[0]
        mask, before = eng.covered_mask(cur), eng.grid_cells()
        removed = eng.remove_covered(cur)
        last[(mask > 0) & (before > 0)] = t
        assert removed == int(before[mask > 0].sum())
        if hl is not None:
            hl = hl[mask[cell_of(hl, gi["nx"], gi["dx"])] == 0]
        if t >= 2 and len(boxes):
            rule(cur, r_max, boxes, h_focus, h_max)
        setp(r_max, cur)
        X0 = model_starts(synth, cur, t, S, spread, g, seed)
        assert np.array_equal(table_b(X0, g), libm_b(X0, g))
        Xs, objs, sts = eng.mads_solve_batch(X0, n_iter, g, (seed + (t - 1) * S) % 2**64)
        f = np.where(objs == objs, objs, math.inf)
        k = int(np.argmin(f)) if np.isfinite(f).any() else 0
        cur = Xs[k].copy()
        X.append(cur)
        obj.append(eng.eval_batch(cur[None, :], want_count=False, want_feasible=False)["obj"][0])
        st.append([k, int(sts["evaluations"].sum()), int(np.isfinite(objs).sum()), removed, appended])
    return np.array(X), np.array(obj), np.array(st, dtype=np.int64), r_max, last, hl


def same_handles(cov, a, b, X, x0, nondyadic=True):
    """Cell store, statistics, classes and 1000 evaluations alike; then one non-dyadic entry added on both (the
    ordered kernel walks each handle's list) and 1000 evaluations alike again."""
    assert np.array_equal(a.grid_cells(), b.grid_cells())
    assert a.grid_info() == b.grid_info()
    assert a.class_weights() == b.class_weights()
    N = x0.size // 3
    C = cov.synth.random_candidates(1000, N, seed=11)
    C[:3] = X[-1], X[0], x0
    for k in ("obj", "count", "feasible"):
        assert np.array_equal(a.eval_batch(C)[k], b.eval_batch(C)[k]), k
    if nondyadic and a.grid_info()["n_classes"] < 4:
        empty = np.flatnonzero(a.grid_cells() == 0)
        p = centres(empty[len(empty) // 2:len(empty) // 2 + 1], a.grid_info()["nx"])
        p[:, 3] = 0.1
        a.add_points(p)
        b.add_points(p)
        assert a.grid_info()["area_exact"] == 0
        ea, eb = a.eval_batch(C), b.eval_batch(C)
        for k in ("obj", "count", "feasible"):
            assert np.array_equal(ea[k], eb[k]), k


def _params(eng, N, sep=0.0):
    def setp(r, prev):
        eng.set_params(N, r, 1e5, prev_xyR=prev, d_lim=10.0, tan_half_fov=T_HALF, sep_min=sep)
    return setp


def _points_scenario(cov, eng, scenario, fire_rows):
    """Store of a scenario on eng; returns (x0, appends, kw)."""
    N = 5
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    kw = dict(S=8, spread=3.0, n_iter=60, granularity=1.0, seed=2**64 - 7, boxes=REF_BOXES, h_focus=15.0, h_max=30.0)
    init = np.concatenate(fire_rows[:10])
    free = np.setdiff1d(np.arange(10000), cell_of(np.concatenate(fire_rows)))  # no fire entry ever lands there
    if scenario.startswith("c5_s"):  # BASELINE C5: rows 1..10, then update_POI's row per timestep
        kw.update(S=int(scenario[4:]), n_iter=100)
        eng.set_points(init, 100, 100, 5.0, 5.0)
        appends = [np.zeros((0, 5))] + [np.asarray(fire_rows[t + 9]) for t in range(2, 41)]
    elif scenario == "refill":  # entries appended onto cells the first timestep emptied, and next to them
        eng.set_grid_full(100, 100, 5.0, 5.0)
        c = np.arange(1, 101) * 5.0 - 2.5
        cx, cy = np.meshgrid(c, c, indexing="ij")
        d = np.min([np.hypot(cx - x0[i], cy - x0[N + i]) - x0[2 * N + i] for i in range(N)], axis=0)
        under = np.flatnonzero((d.T.ravel() < -2.0))
        ring = np.flatnonzero((d.T.ravel() > 0.5) & (d.T.ravel() < 6.0))
        appends = [np.zeros((0, 5))] * 10
        appends[2] = centres(np.concatenate([under[::3], ring[::4]]))
        appends[5] = centres(np.concatenate([under[1::3], under[1::3]]))
        appends[8] = centres(under[::2])
    elif scenario == "pow2":  # multiplicities 1 -> 2 -> 4 far from the swarm: 3 envelope planes, 1 left at the end
        far = np.arange(0, 30)  # row j = 1, x <= 150 m
        eng.set_points(centres(far), 100, 100, 5.0, 5.0)
        appends = [np.zeros((0, 5))] * 6
        appends[1] = centres(far)
        appends[3] = centres(np.concatenate([far, far]))
    elif scenario == "new_weight":  # weight 12.5 first appears mid-horizon
        eng.set_points(init, 100, 100, 5.0, 5.0)
        appends = [np.asarray(fire_rows[t + 9]) if t > 1 else np.zeros((0, 5)) for t in range(1, 9)]
        extra = centres(free[-100::7])
        extra[:, 3] = 12.5
        appends[3] = np.concatenate([appends[3], extra[:8]])
        appends[6] = np.concatenate([extra[8:], appends[6]])
    elif scenario == "grid_full":  # a store without a list: createPOI's order fixed first
        eng.set_grid_full(100, 100, 5.0, 5.0)
        appends = [np.asarray(fire_rows[t]) for t in range(12)]
    elif scenario == "empty":
        eng.set_points(init, 100, 100, 5.0, 5.0)
        appends = [np.zeros((0, 5))] * 8
    setp = _params(eng, N)
    setp(np.full(N, 30 * T_HALF), x0)
    return x0, appends, kw


POINT_SCENARIOS = ["c5_s1", "c5_s148", "refill", "pow2", "new_weight", "grid_full", "empty"]


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", POINT_SCENARIOS)
def test_fire_list_bit_for_bit_against_single_calls(cov, engine, fire_rows, scenario):
    ref = cov.CoverageEngine(0)
    try:
        x0, appends, kw = _points_scenario(cov, engine, scenario, fire_rows)
        _points_scenario(cov, ref, scenario, fire_rows)
        X, obj, st, ms, last = engine.run_horizon_points(x0, appends, **kw)
        T, N = len(appends), x0.size // 3

        def add(t):
            if len(appends[t - 1]):
                ref.add_points(appends[t - 1])
            return len(appends[t - 1])

        Xr, objr, str_, r_end, lastr, _ = replay(cov.synth, ref, x0, T, kw["S"], kw["spread"], kw["n_iter"],
                                                 kw["granularity"], kw["seed"], kw["boxes"], kw["h_focus"],
                                                 kw["h_max"], np.full(N, 30 * T_HALF), _params(ref, N), add)
        assert np.array_equal(X.view(np.uint64), Xr.view(np.uint64)), np.flatnonzero(np.any(X != Xr, axis=1))[:5]
        assert np.array_equal(obj.view(np.uint64), objr.view(np.uint64)), (obj, objr)
        got = np.stack([st[k] for k in ("winner", "evaluations", "feasible", "removed", "appended")], axis=1)
        assert np.array_equal(got, str_), (got, str_)
        assert np.array_equal(last, lastr)
        assert ms.shape == (T,) and np.all(ms > 0)
        if scenario.startswith("c5"):
            assert got[:, 3].sum() > 0 and got[:, 4].sum() == 3474
        if scenario == "refill":  # some entries landed on cells emptied before, some of them survived
            ta = np.concatenate([np.full(len(a), t) for t, a in enumerate(appends, 1)])
            ci = cell_of(np.concatenate(appends))
            hit = (lastr[ci] > 0) & (lastr[ci] < ta)
            assert hit.any() and got[0, 3] > 0
        if scenario == "pow2":
            assert ref.grid_info()["n_planes"] == 1 and ref.grid_cells().max() == 4  # the envelope held bits 0..2
        if scenario == "new_weight":
            assert ref.class_weights()[:2] == [25.0, 12.5]
        if scenario == "empty":  # cov_run_horizon's horizon, with the appended column zero
            third = cov.CoverageEngine(0)
            try:
                _points_scenario(cov, third, scenario, fire_rows)
                Xs, objs, sts, _ = third.run_horizon(x0, T, **kw)
                assert np.array_equal(Xs, X) and np.array_equal(objs, obj) and not got[:, 4].any()
                assert all(np.array_equal(sts[k], st[k]) for k in sts)
            finally:
                third.close()
        same_handles(cov, engine, ref, X, x0)
    finally:
        ref.close()


FIRE_SCHEDULES = {"one_per_step": [0] + [1] * 11, "irregular": [2, 0, 3, 1, 0, 2, 1, 4, 0, 1]}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FIRE_SCHEDULES))
def test_automaton_bit_for_bit_against_single_calls(cov, engine, name):
    steps = FIRE_SCHEDULES[name]
    ref = cov.CoverageEngine(0)
    try:
        N = 5
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 330.0)
        kw = dict(S=16, spread=3.0, n_iter=60, granularity=1.0, seed=41, boxes=REF_BOXES, h_focus=15.0, h_max=30.0)
        fa, fb = cov.DynamicArea.ForestFire(engine, seed=5), cov.DynamicArea.ForestFire(ref, seed=5)
        fa.step()
        fb.step()  # both streams at step 1
        for e in (engine, ref):
            _params(e, N)(np.full(N, 30 * T_HALF), x0)
        X, obj, st, ms = fa.run_horizon(x0, steps, **kw)
        assert fa.t == 1 + sum(steps)

        def burn(t):
            return sum(fb.step() for _ in range(steps[t - 1]))

        Xr, objr, str_, _, _, _ = replay(cov.synth, ref, x0, len(steps), kw["S"], kw["spread"], kw["n_iter"],
                                         kw["granularity"], kw["seed"], kw["boxes"], kw["h_focus"], kw["h_max"],
                                         np.full(N, 30 * T_HALF), _params(ref, N), burn)
        assert np.array_equal(X.view(np.uint64), Xr.view(np.uint64))
        assert np.array_equal(obj.view(np.uint64), objr.view(np.uint64))
        got = np.stack([st[k] for k in ("winner", "evaluations", "feasible", "removed", "appended")], axis=1)
        assert np.array_equal(got, str_), (got, str_)
        assert got[:, 4].sum() > 0 and got[:, 3].sum() > 0
        assert np.array_equal(engine.fire_state(), ref.fire_state()) and fa.t == fb.t
        assert fa.step() == fb.step()  # the same stream continues on both
        assert np.array_equal(engine.fire_state(), ref.fire_state())
        same_handles(cov, engine, ref, X, x0)
    finally:
        ref.close()


# ---------------------------------------------------------------- GPU: refusals change nothing
@pytest.mark.gpu
def test_errors_leave_the_handle_unchanged(cov, engine, fire_rows):
    L = cov._lib
    lib, h = L.lib, engine.handle
    N = 5
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    Xo = np.empty((4, 3 * N))
    B = REF_BOXES.copy()
    none = np.zeros((0, 5))

    def points(appends=(none,) * 4, T=None, S=2, spread=3.0, n_iter=5, g=1.0, xs=x0, X=Xo, boxes=B, nb=1,
               offsets=None, pts="auto"):
        rows = [np.asarray(a, dtype=np.float64).reshape(-1, 5) for a in appends]
        off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64) if offsets is None else offsets
        P = np.ascontiguousarray(np.concatenate(rows)) if rows else none
        pp = (P.ctypes.data if len(P) else None) if isinstance(pts, str) else pts
        return lib.cov_run_horizon_points(h, None if xs is None else xs.ctypes.data, len(rows) if T is None else T, S,
                                          spread, n_iter, g, 0, None if boxes is None else boxes.ctypes.data, nb,
                                          15.0, 30.0, pp, None if off is None or isinstance(off, int) else
                                          off.ctypes.data, None if X is None else X.ctypes.data, None, None, None,
                                          None)

    fs_default = np.array([1, 1, 1, 1], dtype=np.int64)

    def fire(fs=fs_default, T=None, first=1, S=2, spread=3.0, n_iter=5, g=1.0, xs=x0, X=Xo, boxes=B, nb=1):
        return lib.cov_run_horizon_fire(h, None if xs is None else xs.ctypes.data, len(fs) if T is None else T, S,
                                        spread, n_iter, g, 0, None if boxes is None else boxes.ctypes.data, nb, 15.0,
                                        30.0, None if fs is None else fs.ctypes.data, *WIND, 3, first,
                                        None if X is None else X.ctypes.data, None, None, None)

    C = cov.synth.random_candidates(1000, N, seed=2)
    C[0] = x0

    def snapshot():
        return engine.grid_cells(), engine.grid_info(), engine.class_weights(), engine.eval_batch(C)

    def unchanged(s0):
        s1 = snapshot()
        assert np.array_equal(s1[0], s0[0]) and s1[1] == s0[1] and s1[2] == s0[2]
        assert all(np.array_equal(s1[3][k], s0[3][k]) for k in s0[3])

    # store and parameters
    assert points() == L.COV_ERR_STATE and fire() == L.COV_ERR_STATE  # no grid
    init = np.concatenate(fire_rows[:10])
    engine.set_points(init, 100, 100, 5.0, 5.0)
    engine.set_params(N, np.full(N, 30 * T_HALF))
    assert points() == L.COV_ERR_STATE  # cons3 off
    _params(engine, N)(np.full(N, 30 * T_HALF), x0)
    s0 = snapshot()
    # cov_run_horizon's own argument classes
    for bad in (dict(T=-1), dict(S=0), dict(n_iter=-1), dict(xs=None), dict(X=None), dict(spread=-1.0),
                dict(spread=math.nan), dict(g=math.nan), dict(nb=-1), dict(boxes=None)):
        assert points(**bad) == L.COV_ERR_INVALID, bad
        unchanged(s0)
    # offsets, pts5, lattice
    row = centres([5050])
    for bad in (dict(offsets=0), dict(offsets=np.array([1, 1, 1, 1, 1], dtype=np.int64)),
                dict(offsets=np.array([0, 2, 1, 1, 1], dtype=np.int64)), dict(appends=(none, row, none, none), pts=None)):
        assert points(**bad) == L.COV_ERR_INVALID, bad
        unchanged(s0)
    off = row.copy()
    off[0, 0] += 0.5
    assert points(appends=(none, off, none, none)) == L.COV_ERR_OFF_LATTICE
    unchanged(s0)
    nan = row.copy()
    nan[0, 3] = math.nan
    assert points(appends=(none, nan, none, none)) == L.COV_ERR_INVALID
    unchanged(s0)
    free = np.flatnonzero(engine.grid_cells() == 0)[::-1]  # from the far corner
    row = centres(free[:1])
    # two weights on one cell: against the store's class, and across the schedule
    occupied = centres(cell_of(init[:1]))
    occupied[:, 3] = 12.5
    assert points(appends=(none, occupied, none, none)) == L.COV_ERR_INVALID
    unchanged(s0)
    other = row.copy()
    other[:, 3] = 12.5
    assert points(appends=(none, row, other, none)) == L.COV_ERR_INVALID
    unchanged(s0)
    # more than 4 classes; more than 8 planes; a bound over 255
    ws = [centres(free[1 + k:2 + k]) for k in range(4)]
    for k, w in enumerate(ws):
        w[:, 3] = 25.0 / 2 ** (k + 1)
    assert points(appends=(none, ws[0], ws[1], np.concatenate(ws[2:]))) == L.COV_ERR_LIMIT
    unchanged(s0)
    a = np.repeat(centres(free[6:7]), 8, axis=0)  # class 0 up to 8: 4 planes
    b = np.repeat(ws[0], 7, axis=0)           # 12.5 up to 7: 3 planes
    c = np.repeat(ws[1], 2, axis=0)           # 6.25 up to 2: 2 planes
    assert points(appends=(none, a, b, c)) == L.COV_ERR_LIMIT
    unchanged(s0)
    # a bound whose area would depend on the list order (a non-dyadic weight)
    nd = row.copy()
    nd[:, 3] = 0.1
    assert points(appends=(none, none, nd, none)) == L.COV_ERR_STATE
    unchanged(s0)
    # the conservative case: 200 entries on a cell under the swarm (removed at t = 1), 100 more at t = 2
    under = int(cell_of(np.array([[x0[0], x0[N], 0, 0, 0]]))[0])
    engine.add_points(np.repeat(centres([under]), 200, axis=0))
    _params(engine, N)(np.full(N, 30 * T_HALF), x0)
    s1 = snapshot()
    assert points(appends=(none, np.repeat(centres([under]), 100, axis=0), none, none)) == L.COV_ERR_LIMIT
    unchanged(s1)
    # the automaton: no cov_fire_init
    assert fire() == L.COV_ERR_STATE
    unchanged(s1)
    ff = cov.DynamicArea.ForestFire(engine, seed=2)
    _params(engine, N)(np.full(N, 30 * T_HALF), x0)
    s2, st2 = snapshot(), engine.fire_state()
    for bad in (dict(fs=None, T=4), dict(fs=np.array([1, -1, 0, 0], dtype=np.int64)), dict(first=-1),
                dict(first=2**32 - 2, fs=np.array([1, 1, 1, 0], dtype=np.int64)), dict(S=0), dict(X=None)):
        assert fire(**bad) == L.COV_ERR_INVALID, bad
        unchanged(s2)
        assert np.array_equal(engine.fire_state(), st2)
    assert fire(first=2**32 - 3, fs=np.array([1, 1, 1, 0], dtype=np.int64)) == L.COV_OK  # the last step is 2^32 - 1
    # a foreign weight class
    ff = cov.DynamicArea.ForestFire(engine, seed=2)
    w = centres([0])
    w[:, 3] = 12.5
    engine.add_points(w)
    _params(engine, N)(np.full(N, 30 * T_HALF), x0)
    s3, st3 = snapshot(), engine.fire_state()
    assert fire() == L.COV_ERR_STATE
    unchanged(s3)
    assert np.array_equal(engine.fire_state(), st3)
    # still usable
    engine.set_points(init, 100, 100, 5.0, 5.0)
    _params(engine, N)(np.full(N, 30 * T_HALF), x0)
    Xh, obj, st, ms, last = engine.run_horizon_points(x0, [none, row], S=4, boxes=REF_BOXES)
    assert Xh.shape == (2, 3 * N) and np.isfinite(obj).all() and list(st["appended"]) == [0, 1]


# ---------------------------------------------------------------- GPU: run_simulation(starts=S), dynamic
@pytest.mark.gpu
def test_run_simulation_dynamic_equals_the_replay(cov, fire_rows):
    CF, FS, TC = cov.CellFunctions, cov.FullSimulation, cov.TDM_Constraints
    params = FS.SimulationParameters(N_iter=60, seed=23, environment_type="dynamic")
    N, steps, S = params.N, 12, 16
    start = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    cells = CF.initialise_POI(CF.Cells(), "dynamic", fire_rows)
    n_xy = len(cells.fire_point_xy_ccordinates)
    r_max = params.h_max * T_HALF * np.ones(N)
    inp, outp, runtimes, objs = FS.run_simulation(cells, start, TC.cons1, [], N, r_max, params, Nt_sim=steps,
                                                  starts=S, spread=2.0)
    ref = cov.CoverageEngine(0)
    try:
        init = np.concatenate([np.asarray(r).reshape(-1, 5) for r in fire_rows[:10]])
        ref.set_points(init, 100, 100, 5.0, 5.0)
        sched = CF.update_POI_schedule(CF.initialise_POI(CF.Cells(), "dynamic", fire_rows), steps)

        def setp(r, prev):
            ref.set_params(N, r, 1e5, prev_xyR=prev, d_lim=params.d_lim, tan_half_fov=T_HALF)

        setp(params.h_max * T_HALF * np.ones(N), start)

        def add(t):
            if len(sched[t - 1]):
                ref.add_points(sched[t - 1])
            return len(sched[t - 1]), sched[t - 1]

        Xr, objr, _, r_end, _, hl = replay(cov.synth, ref, start, steps, S, 2.0, params.N_iter, 1.0, params.seed,
                                           FS._boxes(params), FS.H_FOCUS, params.h_max,
                                           params.h_max * T_HALF * np.ones(N), setp, add, hl=init)
        assert np.array_equal(np.array(outp), Xr) and np.array_equal(np.array(objs), objr)
        assert np.array_equal(np.array(inp), np.concatenate([start[None], Xr[:-1]]))
        assert len(runtimes) == steps and all(r > 0 for r in runtimes)
        assert np.array_equal(r_max, r_end)
        pl = cells.points_of_interest
        assert np.array_equal(pl.data, hl)  # row for row: update_POI's appends, rmvCoveredPOI's removals
        assert len(cells.fire_point_xy_ccordinates) == n_xy + sum(len(a) for a in sched)
        assert cells.resident()._synced == (id(pl), pl.version)
        eng = cells.resident().engine
        assert np.array_equal(eng.grid_cells(), ref.grid_cells()) and eng.grid_info() == ref.grid_info()
    finally:
        ref.close()
        cells.close()
