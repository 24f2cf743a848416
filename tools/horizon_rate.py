"""Config 1's receding horizon (T = 40 timesteps of FullSimulation's MADS loop) three ways:

  run_simulation   today's driver: per timestep rmvCoveredPOI, the r_max rule, cons3, one cov_mads_solve (Python loop)
  host_loop        the same horizon from existing calls: cov_remove_covered, the rule in NumPy, cov_set_params,
                   cov_mads_solve_batch on S starts, a host argmin and cov_eval_batch per timestep
  run_horizon      cov_run_horizon: all T timesteps enqueued, one synchronise

Config 1: createPOI on 100 x 100 cells of 5 m, N = 5, allocate_even_circles(15, 5, 10 tan 50 deg, 250, 250),
r_max = 30 tan 50 deg, d_lim 10, N_iter 100, granularity 1, the reference's high-interest rectangle, seed 3.
host_loop and run_horizon draw the same starts (spread 3 m) and keys, so at equal S they compute the same horizon.
Per entry: wall time per horizon (host clock around the whole call, median of 5 after one warm-up), the summed
per-timestep device times of run_horizon's step_ms, and the entries covered after 40 timesteps (10000 minus what is
left once the starting swarm and all 40 results have been removed).

    python tools/horizon_rate.py [--out profiles/r5_horizon_rate.json]
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

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import coverage_b200 as cov  # noqa: E402

T_HALF = cov.TAN_HALF_FOV_DEFAULT
N, STEPS, N_ITER, SEED, SPREAD, REPEATS = 5, 40, 100, 3, 3.0, 5
M32 = 0xFFFFFFFF
PARAMS = cov.FullSimulation.SimulationParameters(N_iter=N_ITER, seed=SEED)
BOXES = cov.FullSimulation._boxes(PARAMS)
START = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)


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


def fresh(eng):
    eng.set_grid_full(100, 100, 5.0, 5.0)
    eng.set_params(N, np.full(N, 30 * T_HALF), 1e5, prev_xyR=START, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)


def covered(X):
    with cov.CoverageEngine(0) as e:
        e.set_grid_full(100, 100, 5.0, 5.0)
        e.set_params(N, np.zeros(N))
        for x in [START] + list(X):
            e.remove_covered(x)
        return 10000 - e.grid_info()["n_entries"]


def run_simulation():
    CF, FS = cov.CellFunctions, cov.FullSimulation
    cells = CF.initialise_POI(CF.Cells(), "static")
    try:
        _, outp, runtimes, objs = FS.run_simulation(cells, START, cov.TDM_Constraints.cons1, [], N,
                                                    np.full(N, 30 * T_HALF), PARAMS, Nt_sim=STEPS)
    finally:
        cells.close()
    return np.array(outp), objs, None


def host_loop(eng, S):
    fresh(eng)
    cur, r_max, X, objs = START.copy(), np.full(N, 30 * T_HALF), [], []
    for t in range(1, STEPS + 1):
        eng.remove_covered(cur)
        if t >= 2:
            cov.FullSimulation.apply_r_max_rule(cur, r_max, N, PARAMS, T_HALF)
        eng.set_params(N, r_max, 1e5, prev_xyR=cur, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)
        Xs, o, _ = eng.mads_solve_batch(starts(cur, t, S), N_ITER, 1.0, SEED + (t - 1) * S)
        f = np.where(o == o, o, math.inf)
        cur = Xs[int(np.argmin(f)) if np.isfinite(f).any() else 0].copy()
        X.append(cur)
        objs.append(eng.eval_batch(cur[None, :], want_count=False, want_feasible=False)["obj"][0])
    return np.array(X), objs, None


def run_horizon(eng, S):
    fresh(eng)
    X, objs, _, ms = eng.run_horizon(START, STEPS, S, SPREAD, N_ITER, 1.0, SEED, BOXES, cov.FullSimulation.H_FOCUS,
                                     PARAMS.h_max)
    return X, objs, float(ms.sum())


def measure(fn):
    fn()  # warm-up
    walls, out = [], None
    for _ in range(REPEATS):
        t0 = time.perf_counter()
        out = fn()
        walls.append(time.perf_counter() - t0)
    X, objs, dev_ms = out
    row = {"wall_ms_median": statistics.median(walls) * 1e3, "wall_ms_all": [w * 1e3 for w in walls],
           "entries_covered": int(covered(X)), "last_objective": float(objs[-1])}
    if dev_ms is not None:
        row["step_ms_sum"] = dev_ms
    return row, X


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r5_horizon_rate.json"))
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown", "config": "1 (createPOI 100 x 100 at 5 m, N = 5)", "T": STEPS,
           "N_iter": N_ITER, "spread_m": SPREAD, "seed": SEED,
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
            row, X = measure(lambda: run_horizon(eng, S))
            if S in same:
                row["same_horizon_as_host_loop"] = bool(np.array_equal(X, same[S]))
            out["runs"][f"run_horizon S={S}"] = row
            print("run_horizon", S, json.dumps(row), flush=True)
    finally:
        eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
