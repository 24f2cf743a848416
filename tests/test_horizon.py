"""cov_run_horizon: T timesteps of FullSimulation's MADS loop (rmvCoveredPOI, the r_max rule, cons3 from the current
swarm, S solves, the best as the next swarm) on the device in one call.

CPU: what nvcc built for the two new kernels; the NumPy model of the documented start stream; the table rule for the
initial mesh's exponent against libm's floor(log10(.)).  GPU: every horizon bit for bit against the same horizon built
from existing calls (cov_remove_covered, the rule in NumPy, cov_set_params, cov_mads_solve_batch on the model's
starts, a host argmin, cov_eval_batch), and both handles alike afterwards; the error classes; run_simulation(starts=S).
"""
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
M32 = 0xFFFFFFFF
REF_BOXES = np.array([[2500.0, 3500.0, 1000.0, 2000.0]])  # SimulationParameters' rectangle: outside the 500 m domain
# the host libm's powers of ten as the library's table holds them (std::pow: +Inf beyond 10^308)
P10 = np.array([10.0 ** b if b <= 308 else math.inf for b in range(0, 401)])


# ---------------------------------------------------------------- CPU: the compiled kernels
@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_horizon_kernels_fit_their_launch():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    hz = {k: v for k, v in usage.items() if "horizon_start_kernel" in k or "horizon_commit_kernel" in k}
    assert len(hz) == 2, sorted(hz)
    for k, v in hz.items():
        assert v["LOCAL"] == 0 and v["STACK"] <= 128, (k, v)
        assert v["REG"] * 256 <= 65536, (k, v)  # 256-thread CTAs


# ---------------------------------------------------------------- the model of the documented start stream
def model_starts(synth, cur, t, S, spread, g, seed):
    """Start 0 = cur; start k >= 1: x_i, y_i + spread * z, z the Irwin-Hall(12) normal of the 12 Philox words with
    counter (t, k, j, 3..5), snapped to the mesh when g > 0; R untouched."""
    n = cur.size
    N = n // 3
    X0 = np.repeat(cur[None, :], S, axis=0)
    if S > 1:
        k = np.repeat(np.arange(1, S, dtype=np.uint64), 2 * N)
        j = np.tile(np.arange(2 * N, dtype=np.uint64), S - 1)
        z0 = np.zeros(k.size, dtype=np.uint64)
        s = np.zeros(k.size, dtype=np.uint64)
        for q in range(3):
            for w in synth._philox(z0 + np.uint64(t & M32), k, j, z0 + np.uint64(3 + q), seed & M32, (seed >> 32) & M32):
                s += w
        z = s.astype(np.float64) * 2.0 ** -32 - 6.0
        x = cur[j.astype(np.int64)] + spread * z
        if g > 0:
            x = np.rint(x / g) * g
        X0[1:, :2 * N] = x.reshape(S - 1, 2 * N)
    return X0


def table_b(X, g):
    """The device's exponent of the initial mesh: the largest b >= 0 with 10^b <= target."""
    target = np.maximum(np.maximum(np.abs(X) / 10.0, 1.0), g)
    return np.searchsorted(P10, target, side="right") - 1


def libm_b(X, g):
    """cov_api.cu's initial_mesh: floor(log10(target)) with the C library's log10."""
    return np.array([math.floor(math.log10(max(max(abs(x) / 10.0, 1.0), g))) for x in np.ravel(X)]).reshape(np.shape(X))


def test_start_model(cov):
    synth = cov.synth
    cur = cov.Base_Functions.allocate_even_circles(15.0, 5, 10 * T_HALF, 250.0, 250.0)
    X0 = model_starts(synth, cur, 7, 4000, 3.0, 1.0, 2**64 - 3)
    assert np.array_equal(X0[0], cur) and np.all(X0[:, 10:] == cur[10:])  # start 0 is cur; R never moves
    assert np.all(X0[1:, :10] == np.rint(X0[1:, :10]))  # on the mesh of granularity 1
    d = (model_starts(synth, cur, 7, 4000, 3.0, 0.0, 2**64 - 3) - cur)[1:, :10] / 3.0
    assert abs(d.mean()) < 0.02 and abs(d.std() - 1.0) < 0.02 and np.abs(d).max() <= 6.0  # Irwin-Hall(12)
    # another timestep, another seed: other normals; spread 0: every start is cur
    assert not np.array_equal(model_starts(synth, cur, 8, 4, 3.0, 0.0, 1)[1:], model_starts(synth, cur, 7, 4, 3.0, 0.0, 1)[1:])
    assert np.array_equal(model_starts(synth, cur, 7, 4, 0.0, 0.0, 1), np.repeat(cur[None], 4, axis=0))


@pytest.mark.parametrize("g", [1.0, 0.5, 0.25])
def test_table_exponent_equals_libm_on_mesh_points(g):
    X = np.arange(-round(1e4 / g), round(1e4 / g) + 1) * g
    assert np.array_equal(table_b(X, g), libm_b(X, g))
    powers = 10.0 * P10[:20]  # |x| / 10 exactly a power of ten
    assert np.array_equal(table_b(powers, g), libm_b(powers, g))


# ---------------------------------------------------------------- GPU: against the horizon built from existing calls
def rule(cur, r_max, boxes, h_focus, h_max):
    """FullSimulation.py:80-87 (the same operations as FullSimulation.apply_r_max_rule)."""
    N = cur.size // 3
    for i in range(N):
        if abs(h_focus - cur[2 * N + i] / T_HALF) < 1:
            m = h_max * T_HALF
            near = ((cur[i] < boxes[:, 1] + m) & (cur[i] > boxes[:, 0] - m) &
                    (cur[i + N] < boxes[:, 3] + m) & (cur[i + N] > boxes[:, 2] - m))
            r_max[i] = h_focus * T_HALF if near.any() else h_max * T_HALF


def host_horizon(synth, eng, x_start, T, S, spread, n_iter, g, seed, boxes, h_focus, h_max, r_max, setp):
    """The horizon from existing calls; setp(r_max, prev) = the scenario's cov_set_params."""
    cur, r_max = x_start.copy(), r_max.copy()
    X, obj, st, planes = [], [], [], []
    for t in range(1, T + 1):
        removed = eng.remove_covered(cur)
        planes.append(eng.grid_info()["n_planes"])
        if t >= 2 and len(boxes):
            rule(cur, r_max, boxes, h_focus, h_max)
        setp(r_max, cur)
        X0 = model_starts(synth, cur, t, S, spread, g, seed)
        assert np.array_equal(table_b(X0, g), libm_b(X0, g))  # the device's initial meshes are the host's
        Xs, objs, sts = eng.mads_solve_batch(X0, n_iter, g, (seed + (t - 1) * S) % 2**64)
        f = np.where(objs == objs, objs, math.inf)
        k = int(np.argmin(f)) if np.isfinite(f).any() else 0
        cur = Xs[k].copy()
        X.append(cur)
        obj.append(eng.eval_batch(cur[None, :], want_count=False, want_feasible=False)["obj"][0])
        st.append([k, int(sts["evaluations"].sum()), int(np.isfinite(objs).sum()), removed])
    return np.array(X), np.array(obj), np.array(st, dtype=np.int64), r_max, planes


def _setup(cov, eng, scenario, fire_rows):
    """Store, parameters and horizon settings of a scenario: returns (x_start, r_max, setp, kw)."""
    N, g, n_iter, S, T, spread, boxes = 5, 1.0, 100, 8, 10, 3.0, REF_BOXES
    h_focus, h_max, sep, c7 = 15.0, 30.0, 0.0, False
    nx = 100
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    r_max = np.full(N, 30 * T_HALF)
    if scenario.startswith("c1_s"):
        S, T = int(scenario[4:]), 40
    elif scenario == "box_inside":  # altitude 15: the rule fires, near the box for some UAVs, away for the others
        x0[2 * N:] = 15 * T_HALF
        r_max[:] = 15 * T_HALF
        boxes, T = np.array([[290.0, 350.0, 0.0, 500.0], [2500.0, 3500.0, 1000.0, 2000.0]]), 12
    elif scenario == "rule_edges":  # cur stays (no iterations); UAVs exactly on the rule's strict edges
        m = h_max * T_HALF
        boxes = np.array([[300.0, 350.0, 200.0, 300.0]])
        r16 = 16 * T_HALF
        assert r16 / T_HALF == 16.0
        x0[2 * N:] = [r16, 15 * T_HALF, 15 * T_HALF, 15 * T_HALF, 15 * T_HALF]  # UAV 0: |15 - 16| = 1, not < 1
        x0[1], x0[N + 1] = boxes[0, 0] - m, 250.0    # x == x_LB - m: not near
        x0[2], x0[N + 2] = boxes[0, 1] + m, 250.0    # x == x_UB + m: not near
        x0[3], x0[N + 3] = 320.0, boxes[0, 2] - m    # y == y_LB - m: not near
        x0[4], x0[N + 4] = 320.0, 250.0              # inside: near
        r_max[:] = 20 * T_HALF
        S, T, n_iter, spread, g = 3, 4, 0, 0.0, 0.0  # identical starts: a three-way tie, won by k = 0
    elif scenario == "infeasible":  # cons7 and cons8 fail for every start and every poll point within 3 iterations
        sep, c7 = 15.0, True
        x0 = np.concatenate([250.0 + 5.0 * np.arange(N), np.full(N, 100.0), np.full(N, 25 * T_HALF)])
        r_max[:] = 25 * T_HALF
        S, T, n_iter, spread = 8, 6, 3, 1.0
    elif scenario == "gran_half":
        g = 0.5
    elif scenario == "gran_zero":
        g, n_iter, T = 0.0, 40, 6
        x0 = x0 + 0.01 * np.arange(3 * N)  # off every mesh
    elif scenario == "n1":
        N = 1
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
        r_max = np.full(N, 30 * T_HALF)
    elif scenario == "n64":
        N, nx, S, T, n_iter = 64, 40, 4, 5, 8
        rng = np.random.default_rng(64)
        x0 = np.concatenate([np.rint(rng.random(2 * N) * 200), np.rint(2 + rng.random(N) * 6)])
        r_max = np.full(N, 6.0)
    if scenario == "fire":
        # the fire list (weight 25) with its own duplicates dropped and two more entries on every cell well inside
        # the first swarm: the multiplicity-2 plane empties at step 1 on the host path only
        pts = np.concatenate(fire_rows)
        ci = np.rint((pts[:, 0] + 2.5) / 5).astype(int) - 1 + 100 * (np.rint((pts[:, 1] + 2.5) / 5).astype(int) - 1)
        pts = pts[np.unique(ci, return_index=True)[1]]
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 300.0)
        c = (np.arange(1, 101) * 5.0 - 2.5)
        cx, cy = np.meshgrid(c, c, indexing="ij")
        inside = np.zeros_like(cx, dtype=bool)
        for i in range(N):
            inside |= np.hypot(cx - x0[i], cy - x0[N + i]) < x0[2 * N + i] - 1.0
        extra = np.stack([cx[inside], cy[inside], np.full(inside.sum(), 25.0), np.full(inside.sum(), 25.0),
                          np.zeros(inside.sum())], axis=1)
        eng.set_points(np.concatenate([pts, extra, extra]), 100, 100, 5.0, 5.0)
        assert eng.grid_info()["n_planes"] == 2 and eng.grid_info()["area_exact"] == 1
    else:
        eng.set_grid_full(nx, nx, 5.0, 5.0)
    if scenario == "force_exact":
        eng.set_option(cov.OPT_FORCE_EXACT, 1)

    def setp(r, prev):
        eng.set_params(N, r, 1e5, prev_xyR=prev, d_lim=10.0, tan_half_fov=T_HALF, sep_min=sep, use_cons7=c7)

    setp(r_max, x0)
    return x0, r_max, setp, dict(T=T, S=S, spread=spread, n_iter=n_iter, granularity=g, seed=2**64 - 5,
                                 boxes=boxes, h_focus=h_focus, h_max=h_max)


SCENARIOS = ["c1_s1", "c1_s32", "c1_s300", "box_inside", "rule_edges", "infeasible", "fire", "gran_half", "gran_zero",
             "n1", "n64", "force_exact"]


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", SCENARIOS)
def test_bit_for_bit_against_existing_calls(cov, engine, fire_rows, scenario):
    ref = cov.CoverageEngine(0)
    try:
        x0, r_max, _, kw = _setup(cov, engine, scenario, fire_rows)
        _, _, setp_ref, _ = _setup(cov, ref, scenario, fire_rows)
        X, obj, st, ms = engine.run_horizon(x0, **kw)
        Xr, objr, str_, r_end, planes = host_horizon(cov.synth, ref, x0, kw["T"], kw["S"], kw["spread"], kw["n_iter"],
                                                     kw["granularity"], kw["seed"], kw["boxes"], kw["h_focus"],
                                                     kw["h_max"], r_max, setp_ref)
        assert np.array_equal(X.view(np.uint64), Xr.view(np.uint64)), np.flatnonzero(np.any(X != Xr, axis=1))[:5]
        assert np.array_equal(obj.view(np.uint64), objr.view(np.uint64)), (obj, objr)
        got = np.stack([st[k] for k in ("winner", "evaluations", "feasible", "removed")], axis=1)
        assert np.array_equal(got, str_), (got, str_)
        assert ms.shape == (kw["T"],) and np.all(ms > 0)
        # both handles alike afterwards: store, its statistics, and the parameters of step T
        assert np.array_equal(engine.grid_cells(), ref.grid_cells())
        assert engine.grid_info() == ref.grid_info()
        N = x0.size // 3
        C = cov.synth.random_candidates(1000, N, seed=11)
        C[:3] = X[-1], X[0], x0
        a, b = engine.eval_batch(C), ref.eval_batch(C)
        for k in ("obj", "count", "feasible"):
            assert np.array_equal(a[k], b[k]), k
        if scenario.startswith("c1_s"):
            assert got[:, 3].sum() > 0 and got[:, 2].min() >= 1
        if scenario == "c1_s32":
            assert got[:, 0].max() > 0  # the winner is not always the unperturbed start
        if scenario == "box_inside":
            assert np.any(r_end != 15 * T_HALF)  # the rule moved some r_max
        if scenario == "rule_edges":
            assert np.array_equal(r_end, np.array([20, 30, 30, 30, 15]) * T_HALF)
            assert np.all(got[:, 0] == 0) and np.all(X == x0)
        if scenario == "infeasible":
            assert np.all(got[:, 2] == 0) and np.all(got[:, 0] == 0) and np.all(X == x0)
        if scenario == "fire":
            assert planes[0] == 1 and engine.grid_info()["n_planes"] == 1  # shrank on the host path at step 1
    finally:
        ref.close()


@pytest.mark.gpu
def test_errors_leave_the_handle_unchanged(cov, engine):
    L = cov._lib
    lib, h = L.lib, engine.handle
    N = 5
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    X = np.empty((4, 3 * N))
    B = REF_BOXES.copy()

    def call(T=4, S=2, spread=3.0, n_iter=5, g=1.0, xs=x0, Xo=X, boxes=B, nb=1):
        return lib.cov_run_horizon(h, None if xs is None else xs.ctypes.data, T, S, spread, n_iter, g, 0,
                                   None if boxes is None else boxes.ctypes.data, nb, 15.0, 30.0,
                                   None if Xo is None else Xo.ctypes.data, None, None, None)

    assert call() == L.COV_ERR_STATE  # no grid
    engine.set_grid_full(100, 100, 5.0, 5.0)
    assert call() == L.COV_ERR_STATE  # no params
    engine.set_params(N, np.full(N, 30 * T_HALF))
    assert call() == L.COV_ERR_STATE  # cons3 off
    engine.set_params(N, np.full(N, 30 * T_HALF), prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF)
    C = cov.synth.random_candidates(500, N, seed=2)
    cells0, info0, ev0 = engine.grid_cells(), engine.grid_info(), engine.eval_batch(C)

    def unchanged():
        assert np.array_equal(engine.grid_cells(), cells0) and engine.grid_info() == info0
        ev = engine.eval_batch(C)
        assert all(np.array_equal(ev[k], ev0[k]) for k in ev0)

    for bad in (dict(T=-1), dict(S=0), dict(S=-3), dict(n_iter=-1), dict(xs=None), dict(Xo=None), dict(spread=-1.0),
                dict(spread=math.inf), dict(spread=math.nan), dict(g=-0.5), dict(g=math.nan), dict(nb=-1),
                dict(boxes=None)):
        assert call(**bad) == L.COV_ERR_INVALID, bad
        unchanged()
    assert call(T=0, xs=None, Xo=None) == L.COV_OK  # nothing to do
    unchanged()
    # the solver's limits, with its wording
    big = np.concatenate([np.full(130, 100.0), np.full(65, 5.0)])
    engine.set_params(65, np.full(65, 30 * T_HALF), prev_xyR=big, d_lim=10.0, tan_half_fov=T_HALF)
    with pytest.raises(cov.CoverageError) as e:
        engine.run_horizon(big, 2)
    assert e.value.code == L.COV_ERR_LIMIT and "64" in e.value.message
    engine.set_grid_full(8192, 8192, 500 / 8192, 500 / 8192)
    engine.set_params(N, np.full(N, 30 * T_HALF), prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF)
    with pytest.raises(cov.CoverageError) as e:
        engine.run_horizon(x0, 2)
    assert e.value.code == L.COV_ERR_LIMIT and "shared memory" in e.value.message
    # a list-order store
    pts = np.array([[2.5, 2.5, 1.0, 0.1, 0.0], [7.5, 2.5, 1.0, 0.3, 0.0]])
    engine.set_points(pts, 100, 100, 5.0, 5.0)
    assert engine.grid_info()["area_exact"] == 0
    engine.set_params(N, np.full(N, 30 * T_HALF), prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF)
    with pytest.raises(cov.CoverageError) as e:
        engine.run_horizon(x0, 2)
    assert e.value.code == L.COV_ERR_STATE
    # still usable
    engine.set_grid_full(100, 100, 5.0, 5.0)
    engine.set_params(N, np.full(N, 30 * T_HALF), prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF)
    assert np.array_equal(engine.eval_batch(C)["obj"], ev0["obj"])
    Xh, obj, st, ms = engine.run_horizon(x0, 3, S=4, boxes=REF_BOXES)
    assert Xh.shape == (3, 3 * N) and np.isfinite(obj).all() and st["removed"][0] > 0


@pytest.mark.gpu
def test_run_simulation_starts_equals_the_host_loop(cov):
    CF, FS, TC = cov.CellFunctions, cov.FullSimulation, cov.TDM_Constraints
    params = FS.SimulationParameters(N_iter=60, seed=23)
    N, steps, S = params.N, 8, 16
    start = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    cells = CF.initialise_POI(CF.Cells(), "static")
    r_max = params.h_max * T_HALF * np.ones(N)
    inp, outp, runtimes, objs = FS.run_simulation(cells, start, TC.cons1, [], N, r_max, params, Nt_sim=steps,
                                                  starts=S, spread=2.0)
    ref = cov.CoverageEngine(0)
    try:
        ref.set_grid_full(100, 100, 5.0, 5.0)
        r0 = params.h_max * T_HALF * np.ones(N)

        def setp(r, prev):
            ref.set_params(N, r, 1e5, prev_xyR=prev, d_lim=params.d_lim, tan_half_fov=T_HALF)

        Xr, objr, _, r_end, _ = host_horizon(cov.synth, ref, start, steps, S, 2.0, params.N_iter, 1.0, params.seed,
                                             FS._boxes(params), FS.H_FOCUS, params.h_max, r0, setp)
        assert np.array_equal(np.array(outp), Xr) and np.array_equal(np.array(objs), objr)
        assert np.array_equal(np.array(inp), np.concatenate([start[None], Xr[:-1]]))
        assert len(runtimes) == steps and all(r > 0 for r in runtimes)
        assert np.array_equal(r_max, r_end)
        # the host list: createPOI's entries whose cells the horizon left
        pl = cells.points_of_interest
        full = cov.AreaCoverageCalculation.createPOI(5.0, 5.0, 100.0, 100.0)
        assert np.array_equal(pl.data, full.data[ref.grid_cells()[full.cell_index()] > 0])
        assert cells.resident()._synced == (id(pl), pl.version)
    finally:
        ref.close()
        cells.close()
    with pytest.raises(ValueError):
        FS.run_simulation(CF.Cells(), start, TC.cons1, [], N, r_max, FS.SimulationParameters(environment_type="dynamic"),
                          Nt_sim=2, starts=4)
    with pytest.raises(ValueError):
        FS.run_simulation(CF.Cells(), start, TC.cons1, [], N, r_max, params, Nt_sim=2, objective="region", starts=4)
