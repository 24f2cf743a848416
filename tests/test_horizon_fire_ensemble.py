"""cov_run_horizon_fire_ensemble: E independent dynamic receding horizons with the device automaton in one call, each
with its own fire realisation, wind and starting swarm, on private copies of the handle's store, parameters and
automaton state.

CPU: what nvcc built for the automaton, which gained a scenario dimension; the refusals that need no device;
ForestFire.run_horizon_ensemble's bookkeeping; the engine wrapper's shape checks.  GPU: every scenario bit for bit
against cov_run_horizon_fire on a twin handle holding the same store, automaton and parameters (X, objectives, all five
stats columns, the cells and the automaton state it leaves); one fire for every scenario with stride 0; the handle is
unchanged, refusals included, and its next cov_fire_step is the one it would have made; the multi-device call against
the single-device one.
"""
import ctypes as C
import math
import os
import re
import shutil
import subprocess
import types

import numpy as np
import pytest

T_HALF = math.tan((100 / 180 * math.pi) / 2)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "maximumareacoverageoptimization.jl_b200", "libcoverage_cuda.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
REF_BOXES = np.array([[2500.0, 3500.0, 1000.0, 2000.0]])  # SimulationParameters' rectangle: outside the 500 m domain
STAT_NAMES = ("winner", "evaluations", "feasible", "removed", "appended")
WIND = (4.0, math.radians(270.0), 0.5)  # ForestFire's defaults: wind speed, direction, prob_spread
# At the defaults every direction probability (4 cos(angle) 0.5 at multiples of 45 deg) is <= 0 or > 1, so the fire does
# not depend on its seed; this wind draws in (0, 1).
STOCHASTIC = (1.0, math.radians(270.0), 0.6)
N = 5


# ---------------------------------------------------------------- CPU
@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_fire_step_kernel_fits_its_launch():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    fs = {k: v for k, v in usage.items() if "fire_step_kernel" in k}
    assert len(fs) == 1, sorted(fs)  # the scenario dimension is a run-time argument, not an instantiation
    for k, v in fs.items():
        assert v["LOCAL"] == 0 and v["STACK"] == 0, (k, v)
        assert v["REG"] * 256 <= 65536, (k, v)  # 256-thread CTAs


def test_refusals_without_a_device(cov):
    L = cov._lib
    lib = L.lib
    x = np.zeros(3 * N)
    X = np.empty(3 * N)
    fs = np.ones(1, dtype=np.int64)
    w = np.array(WIND)
    assert lib.cov_run_horizon_fire_ensemble(None, x.ctypes.data, 1, 1, 1, 3.0, 10, 1.0, 0, None, 0, 15.0, 30.0,
                                             fs.ctypes.data, w.ctypes.data, 0, 1, 1, X.ctypes.data, None, None, None,
                                             None, None) == L.COV_ERR_INVALID
    assert lib.cov_multi_run_horizon_fire_ensemble(None, x.ctypes.data, 1, 1, 1, 3.0, 10, 1.0, 0, None, 0, 15.0, 30.0,
                                                   fs.ctypes.data, w.ctypes.data, 0, 1, 1, X.ctypes.data, None, None,
                                                   None, None) == L.COV_ERR_INVALID


def test_forest_fire_run_horizon_ensemble_leaves_the_step_stream(cov):
    calls = []
    eng = types.SimpleNamespace(
        fire_init=lambda *a, **k: None,
        run_horizon_fire_ensemble=lambda *a, **k: calls.append(("ensemble", a, k)) or "out",
        run_horizon_fire=lambda *a, **k: calls.append(("horizon", a, k)) or "out",
        fire_step=lambda *a, **k: calls.append(("step", a, k)) or 0)
    ff = cov.DynamicArea.ForestFire(eng, seed=9)
    ff.step()
    ff.step()
    xs = np.zeros((3, 15))
    assert ff.run_horizon_ensemble(xs, [2, 0, 3], S=4) == "out"
    kind, a, k = calls[-1]
    assert kind == "ensemble" and a[0] is xs and list(a[1]) == [2, 0, 3]
    assert a[2] == (ff.wind_speed, ff.wind_direction, ff.prob_spread) and a[3:] == (9, 3)  # this fire's wind, seed, t+1
    assert k == {"fire_seed_stride": 1, "S": 4} and ff.t == 2  # the engine's fire has not moved
    winds = np.ones((3, 3))
    ff.run_horizon_ensemble(xs, [1], winds=winds, fire_seed_stride=0, want_states=True)
    _, a, k = calls[-1]
    assert a[2] is winds and a[4] == 3 and k == {"fire_seed_stride": 0, "want_states": True} and ff.t == 2
    ff.step()
    assert calls[-1][0] == "step" and calls[-1][1][4] == 3  # step() continues where it was


def test_engine_shape_errors(cov):
    eng = cov.CoverageEngine.__new__(cov.CoverageEngine)  # no device: every check comes before the library call
    eng._h, eng.N = None, N
    xs = np.zeros((2, 3 * N))
    for bad in (dict(x_starts=np.zeros((2, 14))), dict(x_starts=np.zeros((2, 2, 3 * N))),
                dict(winds=np.zeros((3, 3))), dict(winds=np.zeros(2)), dict(winds=np.zeros((2, 4)))):
        kw = dict(x_starts=xs, fire_steps=[1, 1], winds=WIND, fire_seed=0, first_step=1)
        kw.update(bad)
        with pytest.raises(ValueError):
            eng.run_horizon_fire_ensemble(**kw)
    eng.N = None
    with pytest.raises(ValueError):  # no set_params yet
        eng.run_horizon_fire_ensemble(xs, [1], WIND, 0, 1)


# ---------------------------------------------------------------- GPU: against cov_run_horizon_fire on a twin handle
def _params(eng, r_max, prev):
    eng.set_params(N, r_max, 1e5, prev_xyR=prev, d_lim=10.0, tan_half_fov=T_HALF)


def _prep(cov, eng, case):
    """The case's fire, store and parameters on eng.  Returns (ForestFire, x_starts (E, 3N), winds (E, 3),
    fire_steps, stride, kw of the solver)."""
    rng = np.random.default_rng(sum(map(ord, case)))
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 330.0)
    E, S, T, n_iter, stride, pre = 3, 4, 10, 60, 1, 0
    steps = None
    winds = np.repeat(np.array(WIND)[None], 3, axis=0)
    starts = None
    ff = cov.DynamicArea.ForestFire(eng, seed=0 if case == "e1_t40" else sum(map(ord, case)) % 17)
    if case == "e1_t40":  # the default ForestFire, one step per timestep from t = 2
        E, S, T, n_iter = 1, 1, 40, 100
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    elif case == "e3_s4_same_starts":  # only the keys and the fire seeds tell the scenarios apart
        starts = np.repeat(x0[None], 3, axis=0)
        winds = np.repeat(np.array([STOCHASTIC]), 3, axis=0)
    elif case == "winds":
        E, T = 4, 8
        winds = np.array([WIND, STOCHASTIC, (4.0, math.radians(270.0), 0.0), (2.0, 0.3, 0.45)])
    elif case == "irregular":
        steps, pre = [2, 0, 3, 1, 0, 2, 1, 4, 0, 1], 2
    elif case == "e148_s1":
        E, S, T, n_iter = 148, 1, 5, 40
    elif case == "e300_s2":  # more scenarios than one wave of persistent CTAs
        E, S, T, n_iter = 300, 2, 4, 30
    elif case == "multi_plane":  # multiplicities above 1 already: a wider envelope
        ci = np.array([5050, 5051, 3070, 6020])
        i, j = ci % 100 + 1, ci // 100 + 1
        pts = np.stack([(i - 0.5) * 5.0, (j - 0.5) * 5.0, np.zeros(4), np.full(4, 25.0), np.zeros(4)], axis=1)
        eng.add_points(np.repeat(pts, [3, 20, 1, 6], axis=0))
        assert eng.grid_cells().max() >= 20
    elif case == "force_exact":
        eng.set_option(cov.OPT_FORCE_EXACT, 1)
    for _ in range(pre):
        ff.step()
    if steps is None:
        steps = [0] + [1] * (T - 1)
    if starts is None:  # distinct starts: moved by up to 40 m, scenario 0 unmoved
        starts = np.repeat(x0[None], E, axis=0)
        starts[1:, :2 * N] += np.rint(rng.uniform(-40, 40, size=(E - 1, 2 * N)))
    if winds.shape[0] != E:
        winds = np.repeat(winds[:1], E, axis=0)
    _params(eng, np.full(N, 30 * T_HALF), x0)
    kw = dict(S=S, spread=3.0, n_iter=n_iter, granularity=1.0, seed=2**64 - 5, boxes=REF_BOXES, h_focus=15.0,
              h_max=30.0)
    return ff, starts, winds, np.array(steps, dtype=np.int64), stride, kw


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _snapshot(cov, eng, seed=11):
    C_ = cov.synth.random_candidates(1000, N, seed=seed)
    return C_, (eng.grid_cells(), eng.grid_info(), eng.class_weights(), eng.eval_batch(C_), eng.fire_state())


def _same_snapshot(eng, C_, snap):
    cells, info, cw, ev, state = snap
    assert np.array_equal(eng.grid_cells(), cells)
    assert eng.grid_info() == info and eng.class_weights() == cw
    assert np.array_equal(eng.fire_state(), state)
    now = eng.eval_batch(C_)
    for k in ev:
        assert np.array_equal(np.asarray(now[k]).view(np.uint8), np.asarray(ev[k]).view(np.uint8)), k


CASES = ["e1_t40", "e3_s4_same_starts", "winds", "irregular", "e148_s1", "e300_s2", "multi_plane", "force_exact"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_every_scenario_equals_cov_run_horizon_fire(cov, engine, case):
    ref = cov.CoverageEngine(0)
    try:
        ff, starts, winds, fs, stride, kw = _prep(cov, engine, case)
        E, T, S, seed = starts.shape[0], len(fs), kw["S"], kw["seed"]
        t0 = ff.t
        C_, snap = _snapshot(cov, engine)
        launches = engine.launch_count()
        X, obj, st, ms, cells, states = ff.run_horizon_ensemble(starts, fs, winds, fire_seed_stride=stride,
                                                                want_cells=True, want_states=True, **kw)
        assert engine.launch_count() - launches == 1 + int(fs.sum()) + 6 * T  # one launch per step for all E
        assert ff.t == t0
        assert X.shape == (E, T, 3 * N) and obj.shape == (E, T) and ms.shape == (T,) and np.all(ms > 0)
        assert cells.shape == states.shape == (E, 10000)
        _same_snapshot(engine, C_, snap)  # the handle is unchanged
        for e in range(E):
            rf, _, _, _, _, _ = _prep(cov, ref, case)
            assert rf.t == t0
            Xr, objr, str_, _ = ref.run_horizon_fire(starts[e], fs, *winds[e], (rf.seed + e * stride) % 2**64, t0 + 1,
                                                     **dict(kw, seed=(seed + e * T * S) % 2**64))
            assert np.array_equal(_bits(X[e]), _bits(Xr)), (e, np.flatnonzero(np.any(X[e] != Xr, axis=1))[:5])
            assert np.array_equal(_bits(obj[e]), _bits(objr)), (e, obj[e], objr)
            for k in STAT_NAMES:
                assert np.array_equal(st[k][e], str_[k]), (e, k, st[k][e], str_[k])
            assert np.array_equal(cells[e], ref.grid_cells()), e
            assert np.array_equal(states[e], ref.fire_state()), e
        assert st["appended"].sum() > 0 and st["removed"].sum() > 0
        if case == "e3_s4_same_starts":  # the keys really are per scenario
            app = st["appended"]
            assert not np.array_equal(app[0], app[1]) and not np.array_equal(app[1], app[2])
        if case == "winds":  # no spread: nothing appended, the state as it started
            assert np.all(st["appended"][2] == 0) and np.array_equal(states[2], snap[4])
            assert st["appended"][1].sum() > 0 and st["appended"][3].sum() > 0
    finally:
        ref.close()


@pytest.mark.gpu
def test_one_fire_for_every_scenario_with_stride_zero(cov, engine):
    ff, starts, winds, fs, _, kw = _prep(cov, engine, "winds")
    winds = np.repeat(np.array([STOCHASTIC]), starts.shape[0], axis=0)
    X, obj, st, ms, states = ff.run_horizon_ensemble(starts, fs, winds, fire_seed_stride=0, want_states=True, **kw)
    assert np.all(states == states[0]) and np.all(st["appended"] == st["appended"][0])  # the fire ignores the swarm
    assert st["appended"].sum() > 0 and not np.array_equal(X[0], X[1])
    _, _, st1, _, states1 = ff.run_horizon_ensemble(starts, fs, winds, fire_seed_stride=1, want_states=True, **kw)
    assert np.array_equal(states1[0], states[0]) and not np.array_equal(states1[1], states[0])  # stride 1: other fires


@pytest.mark.gpu
def test_handle_unchanged_and_next_step(cov, engine):
    twin = cov.CoverageEngine(0)
    try:
        ff, starts, winds, fs, stride, kw = _prep(cov, engine, "irregular")
        ft, _, _, _, _, _ = _prep(cov, twin, "irregular")
        C_, snap = _snapshot(cov, engine)
        X, obj, st, ms = ff.run_horizon_ensemble(starts, fs, winds, **kw)
        assert st["appended"].sum() > 0
        _same_snapshot(engine, C_, snap)
        _same_snapshot(twin, C_, snap)
        a, b = ff.step(), ft.step()
        assert a == b > 0  # the next step is the one the handle would have made
        _same_snapshot(engine, C_, _snapshot(cov, twin)[1])
    finally:
        twin.close()


@pytest.mark.gpu
def test_refusals_leave_the_handle_unchanged(cov, engine):
    L = cov._lib
    lib, h = L.lib, engine.handle
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 330.0)
    xs = np.stack([x0, x0])
    Xo = np.empty((2, 4, 3 * N))
    fs4 = np.array([0, 1, 1, 1], dtype=np.int64)
    w2 = np.array([WIND, WIND])

    def call(E=2, T=4, S=2, fs=fs4, w=w2, first=1, Xo_=Xo):
        return lib.cov_run_horizon_fire_ensemble(h, xs.ctypes.data, E, T, S, 3.0, 5, 1.0, 0, REF_BOXES.ctypes.data, 1,
                                                 15.0, 30.0, None if fs is None else fs.ctypes.data,
                                                 None if w is None else w.ctypes.data, 3, 1, first,
                                                 None if Xo_ is None else Xo_.ctypes.data, None, None, None, None, None)

    # no cov_fire_init
    engine.set_grid_full(100, 100, 5.0, 5.0)
    _params(engine, np.full(N, 30 * T_HALF), x0)
    C0, s0 = cov.synth.random_candidates(1000, N, seed=3), None
    s0 = (engine.grid_cells(), engine.grid_info(), engine.eval_batch(C0)["obj"])
    assert call() == L.COV_ERR_STATE
    assert np.array_equal(engine.grid_cells(), s0[0]) and engine.grid_info() == s0[1]
    assert np.array_equal(engine.eval_batch(C0)["obj"], s0[2])
    # cons3 off
    cov.DynamicArea.ForestFire(engine, seed=2)
    engine.set_params(N, np.full(N, 30 * T_HALF))
    C_, snap = _snapshot(cov, engine)
    assert call() == L.COV_ERR_STATE
    _same_snapshot(engine, C_, snap)
    # the arguments
    _params(engine, np.full(N, 30 * T_HALF), x0)
    C_, snap = _snapshot(cov, engine)
    for bad in (dict(fs=None), dict(fs=np.array([1, -1, 0, 0], dtype=np.int64)), dict(w=None), dict(E=0),
                dict(E=-1), dict(E=2**30, S=2), dict(first=-1), dict(first=2**32 - 2), dict(Xo_=None), dict(S=0)):
        assert call(**bad) == L.COV_ERR_INVALID, bad
        _same_snapshot(engine, C_, snap)
    assert call(T=0, fs=None, w=None) == L.COV_OK  # nothing to do
    _same_snapshot(engine, C_, snap)
    # an envelope over 255: 250 entries on an interior TREE cell (+ 8)
    tree = int(np.flatnonzero(engine.fire_state().reshape(100, 100)[1:-1, 1:-1].ravel() == 1)[0])
    jj, ii = divmod(tree, 98)
    pt = np.array([[(ii + 1.5) * 5.0, (jj + 1.5) * 5.0, 0.0, 25.0, 0.0]])
    engine.add_points(np.repeat(pt, 250, axis=0))
    _params(engine, np.full(N, 30 * T_HALF), x0)
    C_, snap = _snapshot(cov, engine)
    assert call() == L.COV_ERR_LIMIT
    _same_snapshot(engine, C_, snap)
    # a second weight class
    cov.DynamicArea.ForestFire(engine, seed=2)
    engine.add_points(np.array([[2.5, 2.5, 0.0, 12.5, 0.0]]))
    _params(engine, np.full(N, 30 * T_HALF), x0)
    C_, snap = _snapshot(cov, engine)
    assert call() == L.COV_ERR_STATE
    _same_snapshot(engine, C_, snap)
    # still usable
    cov.DynamicArea.ForestFire(engine, seed=2)
    _params(engine, np.full(N, 30 * T_HALF), x0)
    assert call() == L.COV_OK and np.isfinite(Xo).all()


def _multi_check(cov, engine, devices):
    lib = cov._lib.lib
    ff, starts, winds, fs, stride, kw = _prep(cov, engine, "winds")
    starts = np.concatenate([starts, starts[::-1], starts[:1]])  # 9 scenarios: uneven shards
    winds = np.concatenate([winds, winds[::-1], winds[:1]])
    E, n, T = starts.shape[0], starts.shape[1], len(fs)
    X, obj, st, _, cells, states = ff.run_horizon_ensemble(starts, fs, winds, want_cells=True, want_states=True, **kw)
    devs = (C.c_int * len(devices))(*devices)
    m = C.c_void_p()
    assert lib.cov_multi_create(devs, len(devices), C.byref(m)) == 0
    shards = []
    try:
        for k in range(len(devices)):
            sh = cov.CoverageEngine.__new__(cov.CoverageEngine)
            sh._h, sh._pinned, sh.N, sh.device, sh.param_owner = C.c_void_p(lib.cov_multi_handle(m, k)), [], None, devices[k], None
            shards.append(sh)
            _prep(cov, sh, "winds")
        Xm, om = np.empty((E, T, n)), np.empty((E, T))
        sm, cm, stm = np.empty((E, T, 5), dtype=np.int64), np.empty_like(cells), np.empty_like(states)
        B = kw["boxes"]
        winds = np.ascontiguousarray(winds)
        assert lib.cov_multi_run_horizon_fire_ensemble(m, starts.ctypes.data, E, T, kw["S"], kw["spread"], kw["n_iter"],
                                                       kw["granularity"], kw["seed"], B.ctypes.data, len(B),
                                                       kw["h_focus"], kw["h_max"], fs.ctypes.data, winds.ctypes.data,
                                                       ff.seed, stride, ff.t + 1, Xm.ctypes.data, om.ctypes.data,
                                                       sm.ctypes.data, cm.ctypes.data, stm.ctypes.data) == 0, \
            lib.cov_multi_last_error(m)
        assert np.array_equal(_bits(Xm), _bits(X)) and np.array_equal(_bits(om), _bits(obj))
        assert np.array_equal(sm, np.stack([st[k] for k in STAT_NAMES], axis=2))
        assert np.array_equal(cm, cells) and np.array_equal(stm, states)
    finally:
        for sh in shards:
            sh._h = None
        lib.cov_multi_destroy(m)


@pytest.mark.gpu
def test_multi_device_equals_single_device(cov, engine):
    _multi_check(cov, engine, [0, 0])
