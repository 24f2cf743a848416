"""Config 1's receding horizon (T = 40, S = 1) for E starting deployments, three ways:

  sequential   E cov_run_horizon calls one after the other on one handle (the store and parameters reset before each)
  threads      E handles driven from min(E, 148) host threads, each thread running its share of the scenarios in turn
  ensemble     one cov_run_horizon_ensemble call

Config 1: createPOI on 100 x 100 cells of 5 m, N = 5, r_max = 30 tan 50 deg, d_lim 10, N_iter 100, granularity 1,
spread 3 m, the reference's high-interest rectangle, seed 3.  Scenario e starts from allocate_even_circles(15, 5,
10 tan 50 deg, 250, 250) moved by a seeded offset (scenario 0 unmoved) and runs with seed 3 + e * T * S, so all three
ways compute the same E horizons; the ensemble's bits are checked against the sequential calls in the same run.
Per entry: wall time (host clock around all E horizons, median of 5 after one warm-up), the summed per-timestep device
times of step_ms where the call reports them, and the mean of the entries each scenario covers after 40 timesteps.
Also cov_run_horizon at S = 1 and 148 (tools/horizon_rate.py's rows), with --baseline-tree also from another built
checkout of the repository (e.g. the parent commit's), to show that the single-scenario path did not move.

    python tools/horizon_ensemble_rate.py [--out profiles/r7_horizon_ensemble_rate.json] [--baseline-tree PATH]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

# the checkout whose coverage_b200 is measured: this one, or the --baseline-tree one for its cov_run_horizon rows
ROOT = os.environ.get("HORIZON_RATE_ROOT") or os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import coverage_b200 as cov  # noqa: E402

T_HALF = cov.TAN_HALF_FOV_DEFAULT
N, STEPS, N_ITER, SEED, SPREAD, REPEATS, S = 5, 40, 100, 3, 3.0, 5, 1
PARAMS = cov.FullSimulation.SimulationParameters(N_iter=N_ITER, seed=SEED)
BOXES = cov.FullSimulation._boxes(PARAMS)
START = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
KW = dict(spread=SPREAD, n_iter=N_ITER, granularity=1.0, boxes=BOXES, h_focus=cov.FullSimulation.H_FOCUS,
          h_max=PARAMS.h_max)


def scenario_starts(E):
    X = np.repeat(START[None], E, axis=0)
    X[1:, :2 * N] += np.rint(np.random.default_rng(7).uniform(-40, 40, size=(E - 1, 2 * N)))
    return X


def fresh(eng):
    eng.set_grid_full(100, 100, 5.0, 5.0)
    eng.set_params(N, np.full(N, 30 * T_HALF), 1e5, prev_xyR=START, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)


def covered(eng, x_start, X):
    """Entries one scenario covers: the starting swarm and its 40 results removed from a fresh store."""
    fresh(eng)
    for x in [x_start] + list(X):
        eng.remove_covered(x)
    return 10000 - eng.grid_info()["n_entries"]


def sequential(eng, X0):
    out, ms = [], 0.0
    for e in range(X0.shape[0]):
        fresh(eng)
        X, obj, st, m = eng.run_horizon(X0[e], STEPS, S, seed=SEED + e * STEPS * S, **KW)
        out.append((X, obj, st))
        ms += float(m.sum())
    return out, ms


def threaded(engs, X0):
    E, G = X0.shape[0], len(engs)
    out = [None] * E

    def work(k):
        for e in range(k, E, G):
            fresh(engs[k])
            X, obj, st, _ = engs[k].run_horizon(X0[e], STEPS, S, seed=SEED + e * STEPS * S, **KW)
            out[e] = (X, obj, st)

    th = [threading.Thread(target=work, args=(k,)) for k in range(G)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    return out, None


def ensemble(eng, X0):
    fresh(eng)
    X, obj, st, ms = eng.run_horizon_ensemble(X0, STEPS, S, seed=SEED, **KW)
    return [(X[e], obj[e], {k: v[e] for k, v in st.items()}) for e in range(X0.shape[0])], float(ms.sum())


def measure(fn):
    fn()  # warm-up
    walls, out = [], None
    for _ in range(REPEATS):
        t0 = time.perf_counter()
        out = fn()
        walls.append(time.perf_counter() - t0)
    row = {"wall_ms_median": statistics.median(walls) * 1e3, "wall_ms_all": [w * 1e3 for w in walls]}
    if out[1] is not None:
        row["step_ms_sum"] = out[1]
    return row, out[0]


def same(a, b):
    return all(np.array_equal(x[0].view(np.uint64), y[0].view(np.uint64)) and
               np.array_equal(x[1].view(np.uint64), y[1].view(np.uint64)) and
               all(np.array_equal(x[2][k], y[2][k]) for k in x[2]) for x, y in zip(a, b))


def horizon_rows():
    """cov_run_horizon at S = 1 and 148 from config 1's start (tools/horizon_rate.py's run_horizon rows)."""
    rows = {}
    with cov.CoverageEngine(0) as eng:
        for s in (1, 148):
            def one():
                fresh(eng)
                X, _, _, ms = eng.run_horizon(START, STEPS, s, seed=SEED, **KW)
                return X, float(ms.sum())
            row, _ = measure(one)
            rows[f"cov_run_horizon S={s}"] = row
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r7_horizon_ensemble_rate.json"))
    ap.add_argument("--baseline-tree", default=None, help="another built checkout for the cov_run_horizon rows")
    ap.add_argument("--horizon-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--sizes", default="1,148,1024")
    args = ap.parse_args()
    if args.horizon_only:  # the baseline build's rows, in a process of its own
        print(json.dumps(horizon_rows()))
        return
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown", "config": "1 (createPOI 100 x 100 at 5 m, N = 5)", "T": STEPS, "S": S,
           "N_iter": N_ITER, "spread_m": SPREAD, "seed": SEED,
           "how": f"host clock around all E horizons, median of {REPEATS} after a warm-up", "runs": {}}
    out["cov_run_horizon"] = {"this build": horizon_rows()}
    if args.baseline_tree:
        env = dict(os.environ, HORIZON_RATE_ROOT=os.path.abspath(args.baseline_tree))
        env.pop("COVERAGE_CUDA_LIB", None)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--horizon-only"], env=env, capture_output=True,
                           text=True, check=True)
        out["cov_run_horizon"]["baseline build"] = json.loads(r.stdout.strip().splitlines()[-1])
    print(json.dumps(out["cov_run_horizon"]), flush=True)
    eng = cov.CoverageEngine(0)
    engs = [cov.CoverageEngine(0) for _ in range(148)]
    try:
        for E in [int(v) for v in args.sizes.split(",")]:
            X0 = scenario_starts(E)
            r_seq, res_seq = measure(lambda: sequential(eng, X0))
            r_thr, res_thr = measure(lambda: threaded(engs[:min(E, 148)], X0))
            r_ens, res_ens = measure(lambda: ensemble(eng, X0))
            cov_mean = float(np.mean([covered(eng, X0[e], res_ens[e][0]) for e in range(E)]))
            r_ens["same_bits_as_sequential"] = same(res_ens, res_seq)
            r_thr["same_bits_as_sequential"] = same(res_thr, res_seq)
            row = {"sequential cov_run_horizon": r_seq, f"threads ({min(E, 148)} handles)": r_thr,
                   "cov_run_horizon_ensemble": r_ens, "entries_covered_mean": cov_mean,
                   "speedup_vs_sequential": r_seq["wall_ms_median"] / r_ens["wall_ms_median"],
                   "speedup_vs_threads": r_thr["wall_ms_median"] / r_ens["wall_ms_median"]}
            out["runs"][f"E={E}"] = row
            print(E, json.dumps({k: (v["wall_ms_median"] if isinstance(v, dict) else v) for k, v in row.items()}),
                  flush=True)
    finally:
        eng.close()
        for e in engs:
            e.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
