"""Config C5's dynamic receding horizon (T = 40 timesteps of FullSimulation's MADS loop with update_POI's fire list)
three ways, and the same loop fed by the device forest-fire automaton:

  run_simulation       today's dynamic driver: per timestep update_POI, rmvCoveredPOI, the r_max rule, cons3, one
                       cov_mads_solve (Python loop)
  host_loop            the same horizon from single calls: cov_add_points, cov_remove_covered, the rule in NumPy,
                       cov_set_params, cov_mads_solve_batch on S starts, a host argmin and cov_eval_batch per timestep
  run_horizon_points   cov_run_horizon_points: all T timesteps with their appends enqueued, one synchronise
  run_horizon_fire     cov_run_horizon_fire on the 100 x 100 ForestFire, one automaton step per timestep from t = 2

C5: FirePoints rows 1..10 (455 entries of weight 25) on 100 x 100 cells of 5 m, then row t + 10 at every timestep
t >= 2 (3 474 more entries, largest multiplicity 3: the envelope is the 2 planes the host path uses), N = 5,
allocate_even_circles(15, 5, 10 tan 50 deg, 250, 250), r_max = 30 tan 50 deg, d_lim 10, N_iter 100, granularity 1,
the reference's high-interest rectangle, seed 3.  host_loop and run_horizon_points draw the same starts (spread 3 m)
and keys, so at equal S they compute the same horizon (checked bit for bit in the same run).  Per entry: wall time per
horizon (host clock around the whole call, median of 5 after one warm-up), the summed per-timestep device times of
step_ms, and the entries covered (removed over the 40 timesteps, plus what the last swarm covers at the end).

    python tools/horizon_dynamic_rate.py [--out profiles/r6_horizon_dynamic_rate.json]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import coverage_b200 as cov  # noqa: E402

T_HALF = cov.TAN_HALF_FOV_DEFAULT
N, STEPS, N_ITER, SEED, SPREAD, REPEATS = 5, 40, 100, 3, 3.0, 5
M32 = 0xFFFFFFFF
PARAMS = cov.FullSimulation.SimulationParameters(N_iter=N_ITER, seed=SEED, environment_type="dynamic")
BOXES = cov.FullSimulation._boxes(PARAMS)
START = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
FIRE_ROWS = cov.fire_io.load_fire_rows_npz(os.path.join(ROOT, "tests", "golden", "fire_rows.npz"))
INIT = np.concatenate([np.asarray(r, dtype=np.float64).reshape(-1, 5) for r in FIRE_ROWS[:10]])
APPENDS = [np.zeros((0, 5))] + [np.asarray(FIRE_ROWS[t + 9], dtype=np.float64).reshape(-1, 5)
                                for t in range(2, STEPS + 1)]
KW = dict(spread=SPREAD, n_iter=N_ITER, granularity=1.0, seed=SEED, boxes=BOXES, h_focus=cov.FullSimulation.H_FOCUS,
          h_max=PARAMS.h_max)


def starts(cur, t, S):
    """cov_run_horizon's documented start stream (Philox counter (t, k, j, 3..5), keyed by the seed)."""
    X0 = np.repeat(cur[None, :], S, axis=0)
    if S > 1:
        k = np.repeat(np.arange(1, S, dtype=np.uint64), 2 * N)
        j = np.tile(np.arange(2 * N, dtype=np.uint64), S - 1)
        z0 = np.zeros(k.size, dtype=np.uint64)
        s = np.zeros(k.size, dtype=np.uint64)
        for q in range(3):
            for w in cov.synth._philox(z0 + np.uint64(t), k, j, z0 + np.uint64(3 + q), SEED & M32, SEED >> 32):
                s += w
        x = cur[j.astype(np.int64)] + SPREAD * (s.astype(np.float64) * 2.0 ** -32 - 6.0)
        X0[1:, :2 * N] = np.rint(x).reshape(S - 1, 2 * N)
    return X0


def setp(eng, r_max, prev):
    eng.set_params(N, r_max, 1e5, prev_xyR=prev, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)


def fresh(eng):
    eng.set_points(INIT, 100, 100, 5.0, 5.0)
    setp(eng, np.full(N, 30 * T_HALF), START)


def covered(X):
    """Entries removed over the horizon driven by X (with update_POI's appends), plus what X[-1] covers at the end."""
    with cov.CoverageEngine(0) as e:
        e.set_points(INIT, 100, 100, 5.0, 5.0)
        e.set_params(N, np.zeros(N))
        n = 0
        for t, prev in enumerate([START] + list(X[:-1]), start=1):
            if len(APPENDS[t - 1]):
                e.add_points(APPENDS[t - 1])
            n += e.remove_covered(prev)
        return n + e.remove_covered(X[-1])


def run_simulation():
    CF, FS = cov.CellFunctions, cov.FullSimulation
    cells = CF.initialise_POI(CF.Cells(), "dynamic", FIRE_ROWS)
    try:
        _, outp, _, objs = FS.run_simulation(cells, START, cov.TDM_Constraints.cons1, [], N, np.full(N, 30 * T_HALF),
                                             PARAMS, Nt_sim=STEPS)
    finally:
        cells.close()
    return np.array(outp), objs, None


def host_loop(eng, S):
    fresh(eng)
    cur, r_max, X, objs = START.copy(), np.full(N, 30 * T_HALF), [], []
    for t in range(1, STEPS + 1):
        if len(APPENDS[t - 1]):
            eng.add_points(APPENDS[t - 1])
        eng.remove_covered(cur)
        if t >= 2:
            cov.FullSimulation.apply_r_max_rule(cur, r_max, N, PARAMS, T_HALF)
        setp(eng, r_max, cur)
        Xs, o, _ = eng.mads_solve_batch(starts(cur, t, S), N_ITER, 1.0, SEED + (t - 1) * S)
        f = np.where(o == o, o, math.inf)
        cur = Xs[int(np.argmin(f)) if np.isfinite(f).any() else 0].copy()
        X.append(cur)
        objs.append(eng.eval_batch(cur[None, :], want_count=False, want_feasible=False)["obj"][0])
    return np.array(X), objs, None


def run_horizon_points(eng, S):
    fresh(eng)
    X, objs, _, ms, _ = eng.run_horizon_points(START, APPENDS, S, **KW)
    return X, objs, float(ms.sum())


def run_horizon_fire(eng, S, stats_out):
    ff = cov.DynamicArea.ForestFire(eng, seed=SEED)  # 100 x 100 cells of 5 m, the reference's ignition block
    setp(eng, np.full(N, 30 * T_HALF), START)
    X, objs, st, ms = ff.run_horizon(START, [0] + [1] * (STEPS - 1), S=S, **KW)
    stats_out.update(appended=int(st["appended"].sum()), removed=int(st["removed"].sum()))
    return X, objs, float(ms.sum())


def measure(fn, cover=True):
    fn()  # warm-up
    walls, out = [], None
    for _ in range(REPEATS):
        t0 = time.perf_counter()
        out = fn()
        walls.append(time.perf_counter() - t0)
    X, objs, dev_ms = out
    row = {"wall_ms_median": statistics.median(walls) * 1e3, "wall_ms_all": [w * 1e3 for w in walls],
           "last_objective": float(objs[-1])}
    if cover:
        row["entries_covered"] = int(covered(X))
    if dev_ms is not None:
        row["step_ms_sum"] = dev_ms
    return row, X


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r6_horizon_dynamic_rate.json"))
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown",
           "config": "C5 (FirePoints rows 1..10, then update_POI's row t + 10 per timestep; 100 x 100 at 5 m, N = 5)",
           "T": STEPS, "N_iter": N_ITER, "spread_m": SPREAD, "seed": SEED,
           "entries": {"initial": int(len(INIT)), "appended": int(sum(len(a) for a in APPENDS))},
           "how": f"host clock around one whole horizon, median of {REPEATS} after a warm-up", "runs": {}}
    eng = cov.CoverageEngine(0)
    try:
        row, _ = measure(run_simulation)
        out["runs"]["run_simulation (cov_mads_solve per step)"] = row
        print("run_simulation", json.dumps(row), flush=True)
        same = {}
        for S in (1, 148):
            row, X = measure(lambda: host_loop(eng, S))
            same[S] = X
            out["runs"][f"host_loop S={S}"] = row
            print("host_loop", S, json.dumps(row), flush=True)
        for S in (1, 148, 1024):
            row, X = measure(lambda: run_horizon_points(eng, S))
            if S in same:
                row["same_horizon_as_host_loop"] = bool(np.array_equal(X.view(np.uint64), same[S].view(np.uint64)))
            out["runs"][f"run_horizon_points S={S}"] = row
            print("run_horizon_points", S, json.dumps(row), flush=True)
        for S in (1, 148):
            st = {}
            row, _ = measure(lambda: run_horizon_fire(eng, S, st), cover=False)
            row["entries_appended"], row["entries_removed"] = st["appended"], st["removed"]
            out["runs"][f"run_horizon_fire S={S} (ForestFire 100 x 100, one step per timestep from t = 2)"] = row
            print("run_horizon_fire", S, json.dumps(row), flush=True)
    finally:
        eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
