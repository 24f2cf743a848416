"""cov_run_horizon_ensemble: E independent static receding horizons in one call, each on a private copy of the handle's
store and parameters, one launch per step for the whole ensemble.

CPU: what nvcc built for the scenario kernels and the generalised cell-store kernels; the refusals that need no device;
the Python checks.  GPU: every scenario bit for bit against cov_run_horizon on a twin handle holding the same store and
parameters with seed + e * T * S (X, objectives, all four stats columns, the cells it leaves); a scenario does not depend
on the ensemble around it; the handle is unchanged, refusals included; run_simulation_ensemble against
run_simulation(starts=S); the multi-device call against the single-device one.
"""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

T_HALF = math.tan((100 / 180 * math.pi) / 2)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "maximumareacoverageoptimization.jl_b200", "libcoverage_cuda.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
REF_BOXES = np.array([[2500.0, 3500.0, 1000.0, 2000.0]])  # SimulationParameters' rectangle: outside the 500 m domain
STAT_NAMES = ("winner", "evaluations", "feasible", "removed")


# ---------------------------------------------------------------- CPU: the compiled kernels
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


@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_scenario_kernels_fit_their_launch():
    usage = _usage()
    solve = {k: v for k, v in usage.items() if "scenario_solve_kernel" in k}
    ev = {k: v for k, v in usage.items() if "scenario_eval_kernel" in k}
    assert len(solve) == 2 and len(ev) == 2, (sorted(solve), sorted(ev))  # one per plane mode (single / multi)
    for k, v in solve.items():  # 256 threads, 2 co-resident CTAs per SM (mads_kernel's plan)
        assert v["LOCAL"] == 0 and v["STACK"] <= 128, (k, v)
        assert v["REG"] * 256 * 2 <= 65536, (k, v)
    for k, v in ev.items():  # 256 threads, one warp per scenario
        assert v["LOCAL"] == 0 and v["STACK"] <= 128, (k, v)
        assert v["REG"] * 256 <= 65536, (k, v)
    # the kernels that gained a scenario dimension: no stack, 256-thread CTAs
    for key in ("remove_covered_kernel", "pack_planes_kernel", "thresholds_kernel"):
        ks = [k for k in usage if key in k]
        assert len(ks) == 1, (key, ks)
        v = usage[ks[0]]
        assert v["LOCAL"] == 0 and v["STACK"] == 0 and v["REG"] * 256 <= 65536, (key, v)
    # the single-scenario solver is still exactly the four mads_kernel instantiations
    assert sum("mads_kernel" in k for k in usage) == 4


def test_refusals_without_a_device(cov):
    L = cov._lib
    lib = L.lib
    x = np.zeros(15)
    X = np.empty(15)
    assert lib.cov_run_horizon_ensemble(None, x.ctypes.data, 1, 1, 1, 3.0, 10, 1.0, 0, None, 0, 15.0, 30.0,
                                        X.ctypes.data, None, None, None, None) == L.COV_ERR_INVALID
    assert lib.cov_multi_run_horizon_ensemble(None, x.ctypes.data, 1, 1, 1, 3.0, 10, 1.0, 0, None, 0, 15.0, 30.0,
                                              X.ctypes.data, None, None, None) == L.COV_ERR_INVALID
    FS, CF, TC = cov.FullSimulation, cov.CellFunctions, cov.TDM_Constraints
    start = cov.Base_Functions.allocate_even_circles(15.0, 5, 10 * T_HALF, 250.0, 250.0)
    r_max = np.full(5, 30 * T_HALF)
    with pytest.raises(ValueError):  # static only
        FS.run_simulation_ensemble(CF.Cells(), [start], TC.cons1, 5, r_max,
                                   FS.SimulationParameters(environment_type="dynamic"), Nt_sim=2)
    with pytest.raises(ValueError):  # no scenario
        FS.run_simulation_ensemble(CF.Cells(), [], TC.cons1, 5, r_max, FS.SimulationParameters(), Nt_sim=2)
    with pytest.raises(ValueError):  # the r_max rule needs a rectangle, as for run_simulation(starts=S)
        FS.run_simulation_ensemble(CF.Cells(), [start], TC.cons1, 5, r_max,
                                   FS.SimulationParameters(x_LB=(), x_UB=(), y_LB=(), y_UB=()), Nt_sim=2)


# ---------------------------------------------------------------- GPU: against cov_run_horizon on a twin handle
def _prep(cov, eng, case):
    """Store and parameters of a case on eng; returns (x_starts (E, 3N), kw of run_horizon_ensemble)."""
    N, g, n_iter, S, T, spread, boxes, E = 5, 1.0, 100, 4, 10, 3.0, REF_BOXES, 3
    sep, c7, nx = 0.0, False, 100
    rng = np.random.default_rng(sum(map(ord, case)))
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    r_max = np.full(N, 30 * T_HALF)
    starts = None
    store = "full"
    if case.startswith("c1_e1_s"):  # config 1
        E, S, T = 1, int(case[7:]), 40
    elif case == "e148_s1":
        E, S, T = 148, 1, 8
    elif case == "e300_s2":  # more scenarios than one wave of persistent CTAs
        E, S, T, n_iter = 300, 2, 4, 40
    elif case == "twins":  # identical starts: only the seeds tell the scenarios apart
        E, S = 2, 4
        starts = np.repeat(x0[None], 2, axis=0)
    elif case == "box_some":  # altitude 15 near the box in scenarios 0 and 2, altitude 10 (rule off) in 1 and 3
        E, T, boxes = 4, 8, np.array([[290.0, 350.0, 0.0, 500.0], [2500.0, 3500.0, 1000.0, 2000.0]])
        r_max[:] = 15 * T_HALF
        starts = np.repeat(x0[None], E, axis=0)
        starts[0::2, 2 * N:] = 15 * T_HALF
        starts[1::2, 2 * N:] = 10 * T_HALF
        starts[:, :N] += np.arange(E)[:, None] * 20.0
    elif case == "infeasible_one":  # cons7 + cons8: scenario 1 has no feasible start, the others move
        sep, c7, E, S, T, n_iter, spread = 15.0, True, 3, 8, 6, 3, 1.0
        r_max[:] = 25 * T_HALF
        bad = np.concatenate([250.0 + 5.0 * np.arange(N), np.full(N, 100.0), np.full(N, 25 * T_HALF)])
        good = np.concatenate([150.0 + 40.0 * np.arange(N), np.full(N, 300.0), np.full(N, 25 * T_HALF)])
        starts = np.stack([good, bad, good + np.concatenate([np.full(N, 7.0), np.zeros(2 * N)])])
    elif case == "gran_half":
        g = 0.5
    elif case == "gran_zero":
        g, n_iter, T = 0.0, 40, 6
        x0 = x0 + 0.01 * np.arange(3 * N)
    elif case == "n1":
        N = 1
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
        r_max = np.full(N, 30 * T_HALF)
    elif case == "n64":
        N, nx, S, T, n_iter, E = 64, 40, 4, 5, 8, 3
        x0 = np.concatenate([np.rint(rng.random(2 * N) * 200), np.rint(2 + rng.random(N) * 6)])
        r_max = np.full(N, 6.0)
    elif case == "dyadic_classes":  # two weight classes, multiplicities up to 3: four bit planes
        store = "cells"
    elif case == "force_exact":
        eng.set_option(cov.OPT_FORCE_EXACT, 1)
    if starts is None:  # distinct starts: the case's swarm moved by up to 30 m, R kept
        starts = np.repeat(x0[None], E, axis=0)
        starts[1:, :2 * N] += np.rint(rng.uniform(-30, 30, size=(E - 1, 2 * N)))
    if store == "cells":
        mult = rng.integers(0, 4, size=nx * nx).astype(np.uint8)
        cls = rng.integers(0, 2, size=nx * nx).astype(np.uint8)
        eng.set_grid_cells(mult, nx, nx, 5.0, 5.0, cls=cls, class_weight=[25.0, 50.0])
        info = eng.grid_info()
        assert info["n_planes"] == 4 and info["area_exact"] == 1, info
    else:
        eng.set_grid_full(nx, nx, 5.0, 5.0)
    eng.set_params(N, r_max, 1e5, prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF, sep_min=sep, use_cons7=c7)
    return starts, dict(T=T, S=S, spread=spread, n_iter=n_iter, granularity=g, seed=2**64 - 7, boxes=boxes,
                        h_focus=15.0, h_max=30.0)


def _snapshot(cov, eng, N, seed=11):
    C_ = cov.synth.random_candidates(1000, N, seed=seed)
    ev = eng.eval_batch(C_)
    return C_, (eng.grid_cells(), eng.grid_info(), eng.class_weights(), ev)


def _same_snapshot(eng, C_, snap):
    cells, info, cw, ev = snap
    assert np.array_equal(eng.grid_cells(), cells)
    assert eng.grid_info() == info and eng.class_weights() == cw
    now = eng.eval_batch(C_)
    for k in ev:
        assert np.array_equal(np.asarray(now[k]).view(np.uint8), np.asarray(ev[k]).view(np.uint8)), k


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


CASES = ["c1_e1_s1", "c1_e1_s32", "e3_s4", "e148_s1", "e300_s2", "twins", "box_some", "infeasible_one", "gran_half",
         "gran_zero", "n1", "n64", "dyadic_classes", "force_exact"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_every_scenario_equals_cov_run_horizon(cov, engine, case):
    ref = cov.CoverageEngine(0)
    try:
        starts, kw = _prep(cov, engine, case)
        E, N = starts.shape[0], starts.shape[1] // 3
        T, S, seed = kw["T"], kw["S"], kw["seed"]
        C_, snap = _snapshot(cov, engine, N)
        launches = engine.launch_count()
        X, obj, st, ms, cells = engine.run_horizon_ensemble(starts, want_cells=True, **kw)
        single_plane = engine.grid_info()["n_planes"] == 1
        assert engine.launch_count() - launches == 1 + T * (7 if E == 1 and single_plane else 6)
        assert X.shape == (E, T, 3 * N) and obj.shape == (E, T) and ms.shape == (T,) and np.all(ms > 0)
        assert cells.shape == (E, engine.grid_info()["nx"] * engine.grid_info()["ny"])
        _same_snapshot(engine, C_, snap)  # the handle is unchanged
        for e in range(E):
            _prep(cov, ref, case)
            kw_e = dict(kw, seed=(seed + e * T * S) % 2**64)
            Xr, objr, str_, _ = ref.run_horizon(starts[e], **kw_e)
            assert np.array_equal(_bits(X[e]), _bits(Xr)), (e, np.flatnonzero(np.any(X[e] != Xr, axis=1))[:5])
            assert np.array_equal(_bits(obj[e]), _bits(objr)), (e, obj[e], objr)
            for k in STAT_NAMES:
                assert np.array_equal(st[k][e], str_[k]), (e, k, st[k][e], str_[k])
            assert np.array_equal(cells[e], ref.grid_cells()), e
        if case.startswith("c1_e1"):  # E = 1 is cov_run_horizon with the call's own seed
            assert st["removed"].sum() > 0 and st["feasible"].min() >= 1
        if case == "twins":
            assert not np.array_equal(X[0], X[1])
        if case == "infeasible_one":
            assert np.all(st["feasible"][1] == 0) and np.all(X[1] == starts[1])
            assert st["feasible"][0].sum() > 0 and np.any(X[0] != starts[0])
        if case == "e300_s2":  # a scenario does not depend on the ensemble around it
            for e in (0, 151, 299):
                Xe, oe, se, _ = engine.run_horizon_ensemble(starts[e:e + 1], **dict(kw, seed=(seed + e * T * S) % 2**64))
                assert np.array_equal(_bits(Xe[0]), _bits(X[e])) and np.array_equal(_bits(oe[0]), _bits(obj[e]))
                assert all(np.array_equal(se[k][0], st[k][e]) for k in STAT_NAMES)
    finally:
        ref.close()


@pytest.mark.gpu
def test_handle_unchanged_and_refusals(cov, engine):
    L = cov._lib
    lib, h = L.lib, engine.handle
    N = 5
    twin = cov.CoverageEngine(0)
    try:
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
        starts = np.stack([x0, x0 + np.concatenate([np.full(2 * N, 9.0), np.zeros(N)])])
        X = np.empty((2, 4, 3 * N))

        def call(E=2, T=4, S=2, spread=3.0, n_iter=5, g=1.0, xs=starts, Xo=X, boxes=REF_BOXES, nb=1):
            return lib.cov_run_horizon_ensemble(h, None if xs is None else xs.ctypes.data, E, T, S, spread, n_iter, g,
                                                0, None if boxes is None else boxes.ctypes.data, nb, 15.0, 30.0,
                                                None if Xo is None else Xo.ctypes.data, None, None, None, None)

        assert call() == L.COV_ERR_STATE  # no grid
        for eng in (engine, twin):
            eng.set_grid_full(100, 100, 5.0, 5.0)
        assert call() == L.COV_ERR_STATE  # no params
        for eng in (engine, twin):
            eng.set_params(N, np.full(N, 30 * T_HALF))
        assert call() == L.COV_ERR_STATE  # cons3 off
        hole = np.array([52.5, 77.5, 10.0])  # empties the cells around (52.5, 77.5) on both handles
        for eng in (engine, twin):
            eng.set_params(N, np.full(N, 30 * T_HALF), prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF)
            assert eng.remove_covered(hole) > 0
        C_, snap = _snapshot(cov, engine, N)
        for bad in (dict(T=-1), dict(S=0), dict(n_iter=-1), dict(xs=None), dict(Xo=None), dict(spread=-1.0),
                    dict(spread=math.nan), dict(g=-0.5), dict(nb=-1), dict(boxes=None), dict(E=0), dict(E=-2),
                    dict(E=2**30, S=2), dict(E=2, S=1, T=2**62), dict(E=0, T=0)):
            assert call(**bad) == L.COV_ERR_INVALID, bad
            _same_snapshot(engine, C_, snap)
        assert call(T=0, xs=None, Xo=None) == L.COV_OK  # nothing to do
        _same_snapshot(engine, C_, snap)
        # a run, then the store and the list mirror behave as on a handle that never ran one
        last = engine.last_launch()
        Xe, obj, st, _ = engine.run_horizon_ensemble(starts, 6, S=4, boxes=REF_BOXES)
        assert np.all(st["removed"][:, 0] > 0)
        assert engine.last_launch() == last  # cov_last_launch describes the evaluation before the call
        _same_snapshot(engine, C_, snap)
        pt = np.array([[52.5, 77.5, 1.0, 0.1, 0.0]])  # a non-dyadic weight on an empty cell: the list-order sum
        for eng in (engine, twin):
            eng.add_points(pt)
            assert eng.grid_info()["area_exact"] == 0
        C2 = cov.synth.random_candidates(1000, N, seed=12)
        a, b = engine.eval_batch(C2), twin.eval_batch(C2)
        for k in a:
            assert np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8)), k
        with pytest.raises(cov.CoverageError) as e:  # list-order stores are refused, as by cov_run_horizon
            engine.run_horizon_ensemble(starts, 2)
        assert e.value.code == L.COV_ERR_STATE
        # the solver's limits
        big = np.concatenate([np.full(130, 100.0), np.full(65, 5.0)])
        engine.set_grid_full(100, 100, 5.0, 5.0)
        engine.set_params(65, np.full(65, 30 * T_HALF), prev_xyR=big, d_lim=10.0, tan_half_fov=T_HALF)
        C3, snap3 = _snapshot(cov, engine, 65)
        with pytest.raises(cov.CoverageError) as e:
            engine.run_horizon_ensemble(np.stack([big, big]), 2)
        assert e.value.code == L.COV_ERR_LIMIT and "64" in e.value.message
        _same_snapshot(engine, C3, snap3)
        with pytest.raises(ValueError):
            engine.run_horizon_ensemble(np.zeros((2, 14)), 2)
    finally:
        twin.close()


@pytest.mark.gpu
def test_run_simulation_ensemble_equals_run_simulation(cov):
    CF, FS, TC = cov.CellFunctions, cov.FullSimulation, cov.TDM_Constraints
    params = FS.SimulationParameters(N_iter=60, seed=23)
    N, steps, S = params.N, 6, 4
    base = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    swarms = [base, base + np.concatenate([np.full(N, 20.0), np.full(N, -15.0), np.zeros(N)]), base.copy()]
    cells = CF.initialise_POI(CF.Cells(), "static")
    try:
        r_max = params.h_max * T_HALF * np.ones(N)
        r_keep = r_max.copy()
        pl = cells.points_of_interest
        data0 = pl.data.copy()
        out = FS.run_simulation_ensemble(cells, swarms, TC.cons1, N, r_max, params, Nt_sim=steps, starts=S, spread=2.0)
        assert len(out) == len(swarms)
        assert np.array_equal(r_max, r_keep)  # the caller's r_max
        assert np.array_equal(cells.points_of_interest.data, data0)  # the host list
        assert cells.resident().engine.grid_info()["n_entries"] == len(data0)  # and the resident store
        for e, sw in enumerate(swarms):
            ce = CF.initialise_POI(CF.Cells(), "static")
            try:
                pe = FS.SimulationParameters(N_iter=60, seed=params.seed + e * steps * S)
                ref = FS.run_simulation(ce, sw, TC.cons1, [], N, params.h_max * T_HALF * np.ones(N), pe, Nt_sim=steps,
                                        starts=S, spread=2.0)
            finally:
                ce.close()
            inp, outp, rt, objs = out[e]
            assert np.array_equal(np.array(inp), np.array(ref[0])) and np.array_equal(np.array(outp), np.array(ref[1]))
            assert np.array_equal(_bits(objs), _bits(ref[3]))
            assert len(rt) == steps and all(r > 0 for r in rt)
        assert not np.array_equal(np.array(out[0][1]), np.array(out[2][1]))  # same start, other seed
    finally:
        cells.close()


def _multi_check(cov, engine, devices):
    L = cov._lib
    lib = L.lib
    starts, kw = _prep(cov, engine, "e3_s4")
    starts = np.concatenate([starts, starts[::-1], starts[:1]])  # 7 scenarios: uneven shards
    E, n, T = starts.shape[0], starts.shape[1], kw["T"]
    X, obj, st, _, cells = engine.run_horizon_ensemble(starts, want_cells=True, **kw)
    devs = (C.c_int * len(devices))(*devices)
    m = C.c_void_p()
    assert lib.cov_multi_create(devs, len(devices), C.byref(m)) == 0
    shards = []
    try:
        for k in range(len(devices)):
            sh = cov.CoverageEngine.__new__(cov.CoverageEngine)
            sh._h, sh._pinned, sh.N, sh.device, sh.param_owner = C.c_void_p(lib.cov_multi_handle(m, k)), [], None, devices[k], None
            shards.append(sh)
            _prep(cov, sh, "e3_s4")
        Xm, om = np.empty((E, T, n)), np.empty((E, T))
        sm, cm = np.empty((E, T, 4), dtype=np.int64), np.empty_like(cells)
        B = kw["boxes"]
        assert lib.cov_multi_run_horizon_ensemble(m, starts.ctypes.data, E, T, kw["S"], kw["spread"], kw["n_iter"],
                                                  kw["granularity"], kw["seed"], B.ctypes.data, len(B), kw["h_focus"],
                                                  kw["h_max"], Xm.ctypes.data, om.ctypes.data, sm.ctypes.data,
                                                  cm.ctypes.data) == 0, lib.cov_multi_last_error(m)
        assert np.array_equal(_bits(Xm), _bits(X)) and np.array_equal(_bits(om), _bits(obj))
        assert np.array_equal(sm, np.stack([st[k] for k in STAT_NAMES], axis=2)) and np.array_equal(cm, cells)
    finally:
        for sh in shards:
            sh._h = None
        lib.cov_multi_destroy(m)


@pytest.mark.gpu
def test_multi_device_equals_single_device(cov, engine):
    _multi_check(cov, engine, [0, 0])


@pytest.mark.gpu
def test_multi_device_on_several_gpus(cov, engine):
    n = cov._lib.lib.cov_device_count()
    if n < 2:
        pytest.skip("needs two or more GPUs")
    _multi_check(cov, engine, list(range(n)))
