"""The dynamic receding horizon over the reference's fire list on a list-order store (COV_OPT_LIST_ORDER_HORIZON):
BASELINE C5 with a high-interest rectangle inside the fire (x 200..300 m, y 240..320 m), so that update_POI gives the
entries there the non-dyadic weight (h_max tan(FOV/2))^2 pi, both in the initial list and in the appends.

  device       one cov_run_horizon_points call with list_order=True (T = 40, S = 1 and 148)
  replay       the same horizon from single calls (the test suite's replay: cov_add_points, cov_remove_covered, the
               r_max rule, cov_set_params, cov_mads_solve_batch, the argmin, cov_eval_batch), with that replay's own
               per-timestep checks inside the clock
  host loop    FullSimulation.run_simulation without starts= (the host MADS loop of the reference, S = 1)
  ensembles    E = 148 and 1024 scenarios in one cov_run_horizon_points_ensemble call against E sequential
               cov_run_horizon_points calls (restores between calls outside the clock)

The device and replay horizons are checked to be the same bits in the same run, and so is every ensemble scenario
against its sequential call.  Wall times from the host clock (median of 3 after a warm-up; the sequential E = 1024
loop and the host loop once).

    python tools/horizon_list_order_rate.py [--out profiles/r10_horizon_list_order_rate.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import coverage_b200 as cov  # noqa: E402
from test_horizon_dynamic import replay  # noqa: E402

T_HALF = cov.TAN_HALF_FOV_DEFAULT
N, STEPS, N_ITER, SEED, SPREAD, REPEATS = 5, 40, 100, 3, 3.0, 3
RECT = ([200.0], [300.0], [240.0], [320.0])
PARAMS = cov.FullSimulation.SimulationParameters(N_iter=N_ITER, seed=SEED, environment_type="dynamic")
BOXES = cov.FullSimulation._boxes(PARAMS)
START = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
KW = dict(spread=SPREAD, n_iter=N_ITER, granularity=1.0, boxes=BOXES, h_focus=cov.FullSimulation.H_FOCUS,
          h_max=PARAMS.h_max)
ROWS = cov.fire_io.load_fire_rows_npz(os.path.join(ROOT, "tests", "golden", "fire_rows.npz"))


def cells():
    c = cov.CellFunctions.Cells()
    c.high_interest = RECT
    return cov.CellFunctions.initialise_POI(c, "dynamic", ROWS)


_C = cells()
INIT = _C.points_of_interest.data.copy()
SCHED = cov.CellFunctions.update_POI_schedule(_C, STEPS)
_C.close()


def fresh(eng):
    eng.set_points(INIT, 100, 100, 5.0, 5.0)
    eng.set_params(N, np.full(N, 30 * T_HALF), 1e5, prev_xyR=START, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def timed(fn, repeats=REPEATS, prepare=None):
    if prepare:
        prepare()
    fn()  # warm-up
    walls, out = [], None
    for _ in range(repeats):
        if prepare:
            prepare()
        t0 = time.perf_counter()
        out = fn()
        walls.append(time.perf_counter() - t0)
    return {"wall_ms_median": statistics.median(walls) * 1e3, "wall_ms_all": [w * 1e3 for w in walls]}, out


def horizon_rows(eng, ref, S):
    def device():
        return eng.run_horizon_points(START, SCHED, S=S, seed=SEED, list_order=True, **KW)
    r_dev, (X, obj, st, ms, last) = timed(device, prepare=lambda: fresh(eng))
    r_dev["step_ms_sum"] = float(ms.sum())

    def setp(r, prev):
        ref.set_params(N, r, 1e5, prev_xyR=prev, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)

    def add(t):
        if len(SCHED[t - 1]):
            ref.add_points(SCHED[t - 1])
        return len(SCHED[t - 1])

    def rep():
        return replay(cov.synth, ref, START, STEPS, S, SPREAD, N_ITER, 1.0, SEED, BOXES, KW["h_focus"], KW["h_max"],
                      np.full(N, 30 * T_HALF), setp, add)
    r_rep, (Xr, objr, str_, _, lastr, _) = timed(rep, repeats=1, prepare=lambda: fresh(ref))
    got = np.stack([st[k] for k in ("winner", "evaluations", "feasible", "removed", "appended")], axis=1)
    same = bool(np.array_equal(bits(X), bits(Xr)) and np.array_equal(bits(obj), bits(objr)) and
                np.array_equal(got, str_) and np.array_equal(last, lastr))
    return {"device cov_run_horizon_points": r_dev, "replay from single calls": r_rep,
            "device_same_bits_as_replay": same, "area_exact_at_start": 0,
            "entries_removed": int(st["removed"].sum()), "entries_appended": int(st["appended"].sum()),
            "speedup_vs_replay": r_rep["wall_ms_median"] / r_dev["wall_ms_median"]}


def host_loop():
    c = cells()
    try:
        t0 = time.perf_counter()
        cov.FullSimulation.run_simulation(c, START.copy(), cov.TDM_Constraints.cons1, [], N,
                                          PARAMS.h_max * T_HALF * np.ones(N), PARAMS, Nt_sim=STEPS)
        return {"wall_ms": (time.perf_counter() - t0) * 1e3}
    finally:
        c.close()


def ensemble_rows(eng, E):
    X0 = np.repeat(START[None], E, axis=0)
    X0[1:, :2 * N] += np.rint(np.random.default_rng(7).uniform(-40, 40, size=(E - 1, 2 * N)))

    def ens():
        return eng.run_horizon_points_ensemble(X0, [SCHED], S=1, seed=SEED, want_cells=True, want_last_removed=True,
                                               list_order=True, **KW)
    fresh(eng)
    r_ens, (X, obj, st, ms, cl, last) = timed(ens)
    r_ens["step_ms_sum"] = float(ms.sum())
    busy, same = 0.0, True
    for e in range(E):
        fresh(eng)
        t0 = time.perf_counter()
        Xe, oe, se, _, le = eng.run_horizon_points(X0[e], SCHED, S=1, seed=SEED + e * STEPS, list_order=True, **KW)
        busy += time.perf_counter() - t0
        same &= bool(np.array_equal(bits(Xe), bits(X[e])) and np.array_equal(bits(oe), bits(obj[e])) and
                     all(np.array_equal(se[k], st[k][e]) for k in se) and np.array_equal(le, last[e]) and
                     np.array_equal(eng.grid_cells(), cl[e]))
    return {"cov_run_horizon_points_ensemble": r_ens, "sequential cov_run_horizon_points": {"wall_ms": busy * 1e3},
            "ensemble_same_bits_as_sequential": same, "speedup_vs_sequential": busy * 1e3 / r_ens["wall_ms_median"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r10_horizon_list_order_rate.json"))
    ap.add_argument("--ensembles", default="148,1024")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown",
           "config": "BASELINE C5 (fire rows 1..10 on 100 x 100 at 5 m, row t + 10 appended at t >= 2; N = 5) with the "
                     "high-interest rectangle x 200..300, y 240..320 m: entries inside weigh (h_max tan 50 deg)^2 pi",
           "T": STEPS, "N_iter": N_ITER, "spread_m": SPREAD, "seed": SEED, "initial_entries": len(INIT),
           "initial_nondyadic_entries": int((INIT[:, 3] != 25.0).sum()),
           "how": f"host clock; device and ensemble: median of {REPEATS} after a warm-up; replay, host loop and the "
                  "sequential loops: once after a warm-up where noted", "horizon": {}, "ensembles": {}}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)

    def save():  # after every row, so that a cut-short run keeps what it measured
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    eng, ref = cov.CoverageEngine(0), cov.CoverageEngine(0)
    try:
        for S in (1, 148):
            out["horizon"][f"S={S}"] = row = horizon_rows(eng, ref, S)
            print(S, json.dumps(row), flush=True)
            save()
        out["horizon"]["host loop run_simulation (S=1)"] = host_loop()
        print(json.dumps(out["horizon"]["host loop run_simulation (S=1)"]), flush=True)
        save()
        for E in (int(v) for v in args.ensembles.split(",") if v):
            out["ensembles"][f"E={E} S=1"] = row = ensemble_rows(eng, E)
            print(E, json.dumps(row), flush=True)
            save()
    finally:
        eng.close()
        ref.close()
    save()
    print("wrote", args.out)


if __name__ == "__main__":
    main()
