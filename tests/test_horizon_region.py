"""cov_run_horizon_region: T timesteps of the region objective's receding horizon (the swarm's discs join the covered
set, the r_max rule, cons3 from the current swarm, S region solves, the best as the next swarm) on the device in one
call.

CPU: what nvcc built for the three new kernels; a NumPy restatement of the arc count of the covered set's boundary
against closed forms.  GPU: every horizon bit for bit against the same horizon built from existing calls on a twin
handle (cov_set_region, the rule in NumPy, cov_set_params, cov_mads_solve_batch_region on test_horizon's model starts,
a host argmin, cov_eval_region_batch), the arc counts against the restatement, both handles alike afterwards; the
refusals and the arc limit crossed inside the loop, which leave the handle unchanged; the launch count;
FullSimulation.run_simulation_region.
"""
import math
import os
import re
import subprocess

import numpy as np
import pytest

from test_horizon import CUOBJDUMP, LIB, REF_BOXES, T_HALF, model_starts, rule
from test_region_objective import _covered_set

DOMAIN = (0.0, 0.0, 500.0, 500.0)
TWO_PI = 6.283185307179586


# ---------------------------------------------------------------- CPU: the compiled kernels
@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_cover_kernels_fit_their_launch():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    plan = {"cover_arcs_kernel": (32, 1), "cover_solve_kernel": (256, 2), "cover_eval_kernel": (256, 2)}
    for key, (threads, ctas) in plan.items():
        ks = [k for k in usage if key in k]
        assert len(ks) == 1, (key, ks)
        v = usage[ks[0]]
        assert v["LOCAL"] == 0 and v["STACK"] <= 128, (key, v)
        assert v["REG"] * threads * ctas <= 65536, (key, v)


# ---------------------------------------------------------------- the arc count, restated
def _blocked(cx, cy, R, discs, m, domain):
    """The parameter intervals of circle m that another disc or the outside of the domain covers, wrapped onto
    [0, 2 pi] as the kernels wrap them; None when the whole circle is covered."""
    out = []
    dist = np.hypot(discs[:, 0] - cx, discs[:, 1] - cy)
    near = np.flatnonzero(dist < R + discs[:, 2])  # the others cover nothing of circle m

    def add(phi, alpha):
        a = math.fmod(phi - alpha, TWO_PI)
        if a < 0:
            a += TWO_PI
        e = a + 2 * alpha
        out.extend([(a, TWO_PI), (0.0, e - TWO_PI)] if e > TWO_PI else [(a, e)])

    for j in near:
        xj, yj, Rj = discs[j]
        if j == m:
            continue
        d = math.hypot(xj - cx, yj - cy)
        if d >= R + Rj:
            continue
        if d + R <= Rj:  # inside disc j: covered, unless identical and the lower index
            if d + Rj <= R and m < j:
                continue
            return None
        if d + Rj <= R:
            continue
        c = (R * R + d * d - Rj * Rj) / (2.0 * R * d)
        add(math.atan2(yj - cy, xj - cx), math.acos(max(-1.0, min(1.0, c))))
    x_lo, y_lo, x_hi, y_hi = domain
    for s, phi in ((cy - y_lo, 1.5 * math.pi), (x_hi - cx, 0.0), (y_hi - cy, 0.5 * math.pi), (cx - x_lo, math.pi)):
        if s >= R:
            continue
        if s <= -R:
            return None
        add(phi, math.acos(s / R))
    return out


def arc_count(discs, domain=DOMAIN):
    """Arcs of the boundary of the union of discs (M x 3, R > 0) inside the domain: per circle, the exposed pieces of
    [0, 2 pi] outside the other discs and inside the domain (a piece that crosses angle 0 counts twice)."""
    discs = np.asarray(discs, dtype=np.float64).reshape(-1, 3)
    K = 0
    for m, (cx, cy, R) in enumerate(discs):
        iv = _blocked(cx, cy, R, discs, m, domain)
        if iv is None:
            continue
        pos = 0.0
        for a, b in sorted(iv):
            if a > pos:
                K += 1
            pos = max(pos, b)
        K += pos < TWO_PI
    return K


def test_arc_count_closed_forms():
    assert arc_count(np.zeros((0, 3))) == 0
    assert arc_count([[250, 250, 30]]) == 1                      # one disc inside: its whole circle
    assert arc_count([[200, 250, 30], [230, 250, 30]]) == 3      # two overlapping discs: circle 1's arc crosses angle 0
    assert arc_count([[250, 10, 30]]) == 2                       # crossing the bottom edge: two pieces either side
    assert arc_count([[490, 250, 30]]) == 1                      # crossing the right edge: one piece around angle 0
    assert arc_count([[250, 250, 30], [250, 250, 30]]) == 1      # identical discs: the lower index keeps the circle
    assert arc_count([[250, 250, 30], [255, 250, 10]]) == 1      # a disc inside another adds nothing
    assert arc_count([[250, 250, 1000]]) == 0                    # covering the whole domain
    assert arc_count([[-100, 250, 30]]) == 0                     # outside the domain


# ---------------------------------------------------------------- GPU: against the horizon built from existing calls
def replay(cov, ref, C0, x0, T, S, spread, n_iter, g, seed, boxes, h_focus, h_max, r_max, setp, domain=DOMAIN):
    """The horizon from existing calls.  Returns X, obj, stats (winner, evaluations, feasible, restated arcs), r_max,
    the covered sets and the failure (t, code) of the first cov_set_region that fails, or None."""
    N = x0.size // 3
    cur, r_max, C = x0.copy(), r_max.copy(), np.asarray(C0, dtype=np.float64).reshape(-1, 3)
    X, obj, st, covered = [], [], [], []
    for t in range(1, T + 1):
        C = np.vstack([C, cur.reshape(3, N).T])
        try:
            ref.set_region(*domain, C)
        except cov.CoverageError as e:
            return np.array(X), np.array(obj), np.array(st, dtype=np.int64), r_max, covered, (t, e.code)
        covered.append(C.copy())
        if t >= 2 and len(boxes):
            rule(cur, r_max, boxes, h_focus, h_max)
        setp(r_max, cur)
        X0 = model_starts(cov.synth, cur, t, S, spread, g, seed)
        Xs, objs, sts = ref.mads_solve_batch_region(X0, n_iter, g, (seed + (t - 1) * S) % 2**64)
        f = np.where(objs == objs, objs, math.inf)
        k = int(np.argmin(f)) if np.isfinite(f).any() else 0
        cur = Xs[k].copy()
        X.append(cur)
        obj.append(ref.eval_region_batch(cur[None, :])["obj"][0])
        st.append([k, int(sts["evaluations"].sum()), int(np.isfinite(objs).sum()), arc_count(C[C[:, 2] > 0], domain)])
    return np.array(X), np.array(obj), np.array(st, dtype=np.int64), r_max, covered, None


def _setup(cov, eng, case):
    """Region, parameters and horizon settings of a case: returns (x0, r_max, C0, setp, kw)."""
    N, g, n_iter, S, T, spread, boxes = 5, 1.0, 100, 1, 40, 3.0, REF_BOXES
    sep, c7 = 0.0, False
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    r_max = np.full(N, 30 * T_HALF)
    C0 = np.zeros((0, 3))
    if case.startswith("c1_s"):
        S = int(case[4:])
    elif case.startswith("ring_s"):  # about 100 ring-shaped discs of earlier swarms
        S, T = int(case[6:]), 40
        C0 = _covered_set(np.random.default_rng(7), 100)
        C0[3, 2] = 0.0  # dropped by cov_set_region
    elif case == "box_inside":  # altitude 15: the rule fires, near the box for some UAVs, away for the others
        x0[2 * N:] = 15 * T_HALF
        r_max[:] = 15 * T_HALF
        boxes, T, S = np.array([[290.0, 350.0, 0.0, 500.0], [2500.0, 3500.0, 1000.0, 2000.0]]), 12, 8
    elif case == "cons78":
        sep, c7, S, T = 15.0, True, 8, 10
    elif case == "n1":
        N, S = 1, 8
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
        r_max = np.full(N, 30 * T_HALF)
    elif case == "n64":
        N, S, T, n_iter = 64, 4, 7, 8  # M = 7 x 64 = 448
        rng = np.random.default_rng(64)
        x0 = np.concatenate([np.rint(rng.random(2 * N) * 500), np.rint(5 + rng.random(N) * 15)])
        r_max = np.full(N, 15.0)
    elif case == "gran_zero":
        g, n_iter, T, S = 0.0, 40, 8, 4
        x0 = x0 + 0.01 * np.arange(3 * N)
    elif case == "gran_half":
        g, T, S = 0.5, 10, 4
    elif case == "r_zero":  # one UAV at R = 0: its disc never joins the covered set
        x0[2 * N + 2] = 0.0
        S, T = 4, 12
    elif case == "t_zero":
        T = 0

    def setp(r, prev):
        eng.set_params(N, r, 1e5, prev_xyR=prev, d_lim=10.0, tan_half_fov=T_HALF, sep_min=sep, use_cons7=c7)

    eng.set_region(*DOMAIN, C0)
    setp(r_max, x0)
    return x0, r_max, C0, setp, dict(T=T, S=S, spread=spread, n_iter=n_iter, granularity=g, seed=2**64 - 5,
                                     boxes=boxes, h_focus=15.0, h_max=30.0)


def same_handles(cov, a, b, N, extra=()):
    C = cov.synth.random_candidates(1000, N, seed=11)
    for i, x in enumerate(extra):
        C[i] = x
    ra, rb = a.eval_region_batch(C), b.eval_region_batch(C)
    for k in ("obj", "area", "feasible"):
        assert np.array_equal(ra[k].view(np.uint8), rb[k].view(np.uint8)), k


CASES = ["c1_s1", "c1_s32", "c1_s148", "ring_s1", "ring_s32", "ring_s148", "box_inside", "cons78", "n1", "n64",
         "gran_zero", "gran_half", "r_zero", "t_zero"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_bit_for_bit_against_existing_calls(cov, engine, case):
    ref = cov.CoverageEngine(0)
    try:
        x0, r_max, C0, _, kw = _setup(cov, engine, case)
        _, _, _, setp_ref, _ = _setup(cov, ref, case)
        n0 = engine.launch_count()
        X, obj, st, ms = engine.run_horizon_region(x0, **kw)
        assert engine.launch_count() - n0 == 5 * kw["T"]  # five launches per timestep
        Xr, objr, str_, r_end, covered, failed = replay(cov, ref, C0, x0, kw["T"], kw["S"], kw["spread"], kw["n_iter"],
                                                        kw["granularity"], kw["seed"], kw["boxes"], kw["h_focus"],
                                                        kw["h_max"], r_max, setp_ref)
        assert failed is None
        T, N = kw["T"], x0.size // 3
        assert X.shape == (T, 3 * N) and obj.shape == (T,) and ms.shape == (T,)
        if T:
            assert np.array_equal(X.view(np.uint64), Xr.view(np.uint64)), np.flatnonzero(np.any(X != Xr, axis=1))[:5]
            assert np.array_equal(obj.view(np.uint64), objr.view(np.uint64)), (obj, objr)
            got = np.stack([st[k] for k in ("winner", "evaluations", "feasible", "arcs")], axis=1)
            assert np.array_equal(got, str_), (got, str_)
            assert np.all(ms > 0)
        # both handles alike afterwards: region and parameters of step T
        same_handles(cov, engine, ref, N, [X[-1], X[0], x0] if T else [x0])
        if case.startswith("c1_s") and case != "c1_s1":
            assert got[:, 0].max() > 0  # the winner is not always the unperturbed start
        if case == "box_inside":
            assert np.any(r_end != 15 * T_HALF)
        if case == "r_zero":
            assert np.sum(covered[0][:, 2] > 0) == N - 1
        if case.startswith("ring"):
            assert got[0, 3] > 100
    finally:
        ref.close()


def _near_limit():
    """Discs on a hexagonal lattice in the lower half of the domain, each overlapping its six neighbours with a hole
    between every three (pitch 20, R = 11): six arcs per inner disc, a little under 2048 in all (restated)."""
    rows, cols, p = 15, 24, 20.0
    return np.array([[15.0 + p * c + (p / 2 if r % 2 else 0.0), 15.0 + p * r * math.sqrt(3) / 2, 11.0]
                     for r in range(rows) for c in range(cols)])


def test_near_limit_lattice():
    C = _near_limit()
    assert 2000 < arc_count(C) <= 2048 and len(C) + 22 * 5 <= 512


@pytest.mark.gpu
def test_arc_limit_inside_the_loop_leaves_the_handle_unchanged(cov, engine):
    ref = cov.CoverageEngine(0)
    try:
        C0 = _near_limit()
        N = 5
        x0 = np.concatenate([np.array([60.0, 150.0, 250.0, 350.0, 440.0]), np.full(N, 420.0), np.full(N, 12.0)])
        kw = dict(T=22, S=4, spread=20.0, n_iter=5, granularity=1.0, seed=3, boxes=REF_BOXES, h_focus=15.0,
                  h_max=30.0)
        r_max = np.full(N, 30 * T_HALF)
        for e in (engine, ref):
            e.set_region(*DOMAIN, C0)
            e.set_params(N, r_max, 1e5, prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF)

        def setp(r, prev):
            ref.set_params(N, r, 1e5, prev_xyR=prev, d_lim=10.0, tan_half_fov=T_HALF)

        C = cov.synth.random_candidates(1000, N, seed=5)
        before = engine.eval_region_batch(C)
        with pytest.raises(cov.CoverageError) as e:
            engine.run_horizon_region(x0, **kw)
        _, _, _, _, _, failed = replay(cov, ref, C0, x0, kw["T"], kw["S"], kw["spread"], kw["n_iter"],
                                       kw["granularity"], kw["seed"], kw["boxes"], kw["h_focus"], kw["h_max"], r_max,
                                       setp)
        assert failed is not None and failed[1] == cov._lib.COV_ERR_LIMIT
        assert e.value.code == cov._lib.COV_ERR_LIMIT and f"timestep {failed[0]}:" in e.value.message, e.value.message
        after = engine.eval_region_batch(C)
        for k in before:
            assert np.array_equal(before[k].view(np.uint8), after[k].view(np.uint8)), k
        # still usable: the same horizon, shorter, runs and matches the replay from the untouched region
        engine.run_horizon_region(x0, **dict(kw, T=1))
    finally:
        ref.close()


@pytest.mark.gpu
def test_refusals_leave_the_handle_unchanged(cov, engine):
    L = cov._lib
    lib, h = L.lib, engine.handle
    N = 5
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    X = np.empty((4, 3 * N))
    B = REF_BOXES.copy()

    def call(T=4, S=2, spread=3.0, n_iter=5, g=1.0, xs=x0, Xo=X, boxes=B, nb=1):
        return lib.cov_run_horizon_region(h, None if xs is None else xs.ctypes.data, T, S, spread, n_iter, g, 0,
                                          None if boxes is None else boxes.ctypes.data, nb, 15.0, 30.0,
                                          None if Xo is None else Xo.ctypes.data, None, None, None)

    assert call() == L.COV_ERR_STATE  # no region
    engine.set_region(*DOMAIN, _covered_set(np.random.default_rng(3), 40))
    assert call() == L.COV_ERR_STATE  # no parameters
    engine.set_params(N, np.full(N, 30 * T_HALF))
    assert call() == L.COV_ERR_STATE  # cons3 off
    big = np.concatenate([np.full(130, 100.0), np.full(65, 5.0)])
    engine.set_params(65, np.full(65, 30 * T_HALF), prev_xyR=big, d_lim=10.0, tan_half_fov=T_HALF)
    with pytest.raises(cov.CoverageError) as e:
        engine.run_horizon_region(big, 2)
    assert e.value.code == L.COV_ERR_LIMIT and "64" in e.value.message
    engine.set_params(N, np.full(N, 30 * T_HALF), prev_xyR=x0, d_lim=10.0, tan_half_fov=T_HALF, sep_min=15.0,
                      use_cons7=True)
    C = cov.synth.random_candidates(800, N, seed=2)
    ev0 = engine.eval_region_batch(C)

    def unchanged():
        ev = engine.eval_region_batch(C)
        assert all(np.array_equal(ev[k].view(np.uint8), ev0[k].view(np.uint8)) for k in ev0)

    Xbig = np.empty((100, 3 * N))
    assert call(T=95, Xo=Xbig) == L.COV_ERR_LIMIT  # 40 + 95 x 5 = 515 > 512
    unchanged()
    for bad in (dict(T=-1), dict(S=0), dict(S=-3), dict(n_iter=-1), dict(xs=None), dict(Xo=None), dict(spread=-1.0),
                dict(spread=math.inf), dict(spread=math.nan), dict(g=-0.5), dict(g=math.nan), dict(nb=-1),
                dict(boxes=None)):
        assert call(**bad) == L.COV_ERR_INVALID, bad
        unchanged()
    for v in (math.nan, math.inf):
        xs = x0.copy()
        xs[7] = v
        assert call(xs=xs) == L.COV_ERR_INVALID
        unchanged()
    assert call(T=0, xs=None, Xo=None) == L.COV_OK  # nothing to do
    unchanged()
    assert call(T=94, Xo=Xbig, n_iter=0, spread=0.0) == L.COV_OK  # 40 + 94 x 5 = 510: accepted (the swarm stays)


@pytest.mark.gpu
def test_run_simulation_region_equals_the_replay(cov):
    CF, FS, TC = cov.CellFunctions, cov.FullSimulation, cov.TDM_Constraints
    params = FS.SimulationParameters(N_iter=60, seed=23)
    N, steps, S = params.N, 8, 16
    start = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
    cells = CF.initialise_POI(CF.Cells(), "static")
    r_max = params.h_max * T_HALF * np.ones(N)
    covered_pb = []
    inp, outp, runtimes, objs = FS.run_simulation_region(cells, start, TC.cons1, N, r_max, params, Nt_sim=steps,
                                                         starts=S, spread=2.0, covered_pb=covered_pb)
    ref = cov.CoverageEngine(0)
    try:
        r0 = params.h_max * T_HALF * np.ones(N)

        def setp(r, prev):
            ref.set_params(N, r, 1e5, prev_xyR=prev, d_lim=params.d_lim, tan_half_fov=T_HALF)

        Xr, objr, _, r_end, covered, failed = replay(cov, ref, np.zeros((0, 3)), start, steps, S, 2.0, params.N_iter,
                                                     1.0, params.seed, FS._boxes(params), FS.H_FOCUS, params.h_max, r0,
                                                     setp)
        assert failed is None
        assert np.array_equal(np.array(outp), Xr) and np.array_equal(np.array(objs), objr)
        assert np.array_equal(np.array(inp), np.concatenate([start[None], Xr[:-1]]))
        assert len(runtimes) == steps and all(r > 0 for r in runtimes)
        assert np.array_equal(r_max, r_end)
        assert len(covered_pb) == steps and all(np.array_equal(a, b) for a, b in zip(covered_pb, covered))
    finally:
        ref.close()
        cells.close()
    with pytest.raises(ValueError):
        FS.run_simulation(CF.Cells(), start, TC.cons1, [], N, r_max, params, Nt_sim=2, objective="region", starts=4)
