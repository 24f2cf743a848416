"""The dynamic receding horizon over the reference's fire list (BASELINE C5, T = 40, S = 1) for E scenarios, three ways:

  sequential   E cov_run_horizon_points calls one after the other on one handle; the store and parameters are restored
               before each call outside the clock (only the calls are timed)
  threads      E handles driven from min(E, 148) host threads, each thread running its share of the scenarios in turn;
               every handle is prepared before the clock starts, and the restores between a thread's later scenarios
               are inside it
  ensemble     one cov_run_horizon_points_ensemble call (the handle is left unchanged, so it is prepared once)

C5: rows 1..10 of the committed fire table in the store, row t + 10 appended at timestep t >= 2; N = 5, r_max = 30 tan
50 deg, d_lim 10, N_iter 100, granularity 1, spread 3 m, the reference's high-interest rectangle.  With L = 8 the
schedules are C5's rows shifted by 0, 2, .., 14 rows (forecasts that run ahead of the fire), scenario e on schedule e % 8.
Scenario e starts from allocate_even_circles(15, 5, 10 tan 50 deg, 250, 250) moved by a seeded offset of up to 40 m
(scenario 0 unmoved), with seed 3 + e * T * S, so all three ways compute the same E horizons; the bits (X, objectives,
stats, the cells and last_removed) are checked against the sequential calls in the same run.  Per entry: wall time
(host clock, median of 3 after one warm-up), the summed per-timestep device times of step_ms where the call reports
them, and the mean entries appended and removed per scenario.

Also the single-scenario paths, cov_run_horizon_points at S = 1 and 148 and 100 cov_add_points calls, with
--baseline-tree also from another built checkout of the repository (e.g. the parent commit's), each build in processes
of its own, alternated over several rounds, to show that the single-scenario path did not move.

    python tools/horizon_points_ensemble_rate.py [--out profiles/r9_horizon_points_ensemble_rate.json]
                                                 [--baseline-tree PATH]
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

# the checkout whose coverage_b200 is measured: this one, or the --baseline-tree one for its single-scenario rows
ROOT = os.environ.get("HORIZON_RATE_ROOT") or os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import coverage_b200 as cov  # noqa: E402

T_HALF = cov.TAN_HALF_FOV_DEFAULT
N, STEPS, N_ITER, SEED, SPREAD, REPEATS, S = 5, 40, 100, 3, 3.0, 3, 1
PARAMS = cov.FullSimulation.SimulationParameters(N_iter=N_ITER, seed=SEED, environment_type="dynamic")
BOXES = cov.FullSimulation._boxes(PARAMS)
START = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
KW = dict(spread=SPREAD, n_iter=N_ITER, granularity=1.0, boxes=BOXES, h_focus=cov.FullSimulation.H_FOCUS,
          h_max=PARAMS.h_max)
ROWS = cov.fire_io.load_fire_rows_npz(os.path.join(ROOT, "tests", "golden", "fire_rows.npz"))
INIT = np.concatenate([np.asarray(r).reshape(-1, 5) for r in ROWS[:10]])


def schedule(shift):
    return [np.zeros((0, 5))] + [np.asarray(ROWS[t + 9 + shift]).reshape(-1, 5) for t in range(2, STEPS + 1)]


def scenario_starts(E):
    X = np.repeat(START[None], E, axis=0)
    X[1:, :2 * N] += np.rint(np.random.default_rng(7).uniform(-40, 40, size=(E - 1, 2 * N)))
    return X


def fresh(eng):
    eng.set_points(INIT, 100, 100, 5.0, 5.0)
    eng.set_params(N, np.full(N, 30 * T_HALF), 1e5, prev_xyR=START, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)


def one(eng, x, sched, e, s=S):
    X, obj, st, ms, last = eng.run_horizon_points(x, sched, S=s, seed=SEED + e * STEPS * s, **KW)
    return (X, obj, st, eng.grid_cells(), last), float(ms.sum())


def sequential(eng, X0, scheds, list_of):
    out, ms, busy = [], 0.0, 0.0
    for e in range(X0.shape[0]):
        fresh(eng)
        t0 = time.perf_counter()
        r, m = one(eng, X0[e], scheds[list_of[e]], e)
        busy += time.perf_counter() - t0
        out.append(r)
        ms += m
    return out, ms, busy


def threaded(engs, X0, scheds, list_of):
    E, G = X0.shape[0], len(engs)
    out = [None] * E

    def work(k):
        for i, e in enumerate(range(k, E, G)):
            if i:
                fresh(engs[k])
            out[e], _ = one(engs[k], X0[e], scheds[list_of[e]], e)

    th = [threading.Thread(target=work, args=(k,)) for k in range(G)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    return out, None, None


def ensemble(eng, X0, scheds, list_of):
    X, obj, st, ms, cells, last = eng.run_horizon_points_ensemble(X0, scheds, list_of, S=S, seed=SEED,
                                                                  want_cells=True, want_last_removed=True, **KW)
    return [(X[e], obj[e], {k: v[e] for k, v in st.items()}, cells[e], last[e]) for e in range(X0.shape[0])], \
        float(ms.sum()), None


def measure(fn, prepare=None):
    if prepare:
        prepare()
    fn()  # warm-up
    walls, out = [], None
    for _ in range(REPEATS):
        if prepare:
            prepare()
        t0 = time.perf_counter()
        out = fn()
        walls.append(out[2] if out[2] is not None else time.perf_counter() - t0)
    row = {"wall_ms_median": statistics.median(walls) * 1e3, "wall_ms_all": [w * 1e3 for w in walls]}
    if out[1] is not None:
        row["step_ms_sum"] = out[1]
    return row, out[0]


def same(a, b):
    return all(np.array_equal(x[0].view(np.uint64), y[0].view(np.uint64)) and
               np.array_equal(x[1].view(np.uint64), y[1].view(np.uint64)) and
               all(np.array_equal(x[2][k], y[2][k]) for k in x[2]) and np.array_equal(x[3], y[3]) and
               np.array_equal(x[4], y[4]) for x, y in zip(a, b))


def single_rows():
    """cov_run_horizon_points at S = 1 and 148 from the base swarm, and 100 cov_add_points calls (C5's rows 11..60,
    twice) on the C5 store."""
    rows = {}
    sched = schedule(0)
    with cov.CoverageEngine(0) as eng:
        for s in (1, 148):
            def run():
                fresh(eng)
                t0 = time.perf_counter()
                _, m = one(eng, START, sched, 0, s)
                return None, m, time.perf_counter() - t0
            rows[f"cov_run_horizon_points S={s}"], _ = measure(run)

        def adds():
            fresh(eng)
            t0 = time.perf_counter()
            for k in range(100):
                eng.add_points(np.asarray(ROWS[10 + k % 50]).reshape(-1, 5))
            return None, None, time.perf_counter() - t0
        rows["100 x cov_add_points"], _ = measure(adds)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r9_horizon_points_ensemble_rate.json"))
    ap.add_argument("--baseline-tree", default=None, help="another built checkout for the single-scenario rows")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of this build and the baseline build")
    ap.add_argument("--single-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--runs", default="1:1,148:1,1024:1,1024:8", help="E:L pairs")
    args = ap.parse_args()
    if args.single_only:  # one build's single-scenario rows, in a process of its own
        print(json.dumps(single_rows()))
        return
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown", "config": "BASELINE C5: fire rows 1..10 on 100 x 100 at 5 m, row t + 10 "
           "appended at t >= 2; N = 5", "T": STEPS, "S": S, "N_iter": N_ITER, "spread_m": SPREAD, "seed": SEED,
           "schedules": "L = 1: C5's; L = 8: C5's rows shifted by 2l rows, scenario e on schedule e % 8",
           "how": f"host clock, median of {REPEATS} after a warm-up; sequential: only the calls are timed, the store "
                  "and parameters are restored before each outside the clock; threads: handles prepared before the "
                  "clock, restores between a thread's later scenarios inside it", "runs": {}}
    builds = {"this build": ROOT}
    if args.baseline_tree:
        builds["baseline build"] = os.path.abspath(args.baseline_tree)
    single = {b: [] for b in builds}
    for _ in range(args.rounds):
        for b, tree in builds.items():
            env = dict(os.environ, HORIZON_RATE_ROOT=tree)
            env.pop("COVERAGE_CUDA_LIB", None)
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--single-only"], env=env,
                               capture_output=True, text=True, check=True)
            single[b].append(json.loads(r.stdout.strip().splitlines()[-1]))
    out["single scenario"] = {
        b: {k: {"wall_ms_median_of_rounds": statistics.median(r[k]["wall_ms_median"] for r in rs),
                "wall_ms_per_round": [r[k]["wall_ms_median"] for r in rs]} for k in rs[0]}
        for b, rs in single.items()}
    print(json.dumps(out["single scenario"]), flush=True)
    eng = cov.CoverageEngine(0)
    engs = [cov.CoverageEngine(0) for _ in range(148)]
    try:
        for run in args.runs.split(","):
            E, L = (int(v) for v in run.split(":"))
            X0 = scenario_starts(E)
            scheds = [schedule(2 * l) for l in range(L)]
            list_of = np.arange(E) % L
            G = min(E, 148)

            def prep_threads():
                for k in range(G):
                    fresh(engs[k])
            r_seq, res_seq = measure(lambda: sequential(eng, X0, scheds, list_of))
            r_thr, res_thr = measure(lambda: threaded(engs[:G], X0, scheds, list_of), prepare=prep_threads)
            fresh(eng)
            r_ens, res_ens = measure(lambda: ensemble(eng, X0, scheds, list_of))
            r_ens["same_bits_as_sequential"] = same(res_ens, res_seq)
            r_thr["same_bits_as_sequential"] = same(res_thr, res_seq)
            row = {"sequential cov_run_horizon_points": r_seq, f"threads ({G} handles)": r_thr,
                   "cov_run_horizon_points_ensemble": r_ens,
                   "entries_appended_mean": float(np.mean([r[2]["appended"].sum() for r in res_ens])),
                   "entries_removed_mean": float(np.mean([r[2]["removed"].sum() for r in res_ens])),
                   "speedup_vs_sequential": r_seq["wall_ms_median"] / r_ens["wall_ms_median"],
                   "speedup_vs_threads": r_thr["wall_ms_median"] / r_ens["wall_ms_median"]}
            out["runs"][f"E={E} L={L}"] = row
            print(E, L, json.dumps({k: (v["wall_ms_median"] if isinstance(v, dict) else v) for k, v in row.items()}),
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
