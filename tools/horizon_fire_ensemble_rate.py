"""The dynamic receding horizon with the device automaton (T = 40, S = 1) for E scenarios, three ways:

  sequential   E cov_run_horizon_fire calls one after the other on one handle; the fire, store and parameters are
               restored before each call outside the clock (only the calls are timed)
  threads      E handles driven from min(E, 148) host threads, each thread running its share of the scenarios in turn;
               every handle is prepared before the clock starts, and the restores between a thread's later scenarios
               are inside it
  ensemble     one cov_run_horizon_fire_ensemble call (the handle is left unchanged, so it is prepared once)

The default 100 x 100 ForestFire (seed 3), N = 5, r_max = 30 tan 50 deg, d_lim 10, N_iter 100, granularity 1, spread
3 m, the reference's high-interest rectangle, one automaton step per timestep from t = 2.  Scenario e starts from
allocate_even_circles(15, 5, 10 tan 50 deg, 250, 250) moved by a seeded offset of up to 40 m (scenario 0 unmoved), with
seed 3 + e * T * S and fire seed 3 + e (fire_seed_stride 1: independent fire realisations), so all three ways compute
the same E horizons; the bits (X, objectives, stats, the automaton state left) are checked against the sequential calls
in the same run.  Per entry: wall time (host clock, median of 3 after one warm-up), the summed per-timestep device times
of step_ms where the call reports them, and the mean entries appended and removed per scenario.

Also the single-scenario paths, cov_run_horizon_fire at S = 1 and 148 and 100 cov_fire_step calls, with --baseline-tree
also from another built checkout of the repository (e.g. the parent commit's), each build in processes of its own,
alternated over several rounds, to show that the single-scenario path did not move.

    python tools/horizon_fire_ensemble_rate.py [--out profiles/r8_horizon_fire_ensemble_rate.json] [--baseline-tree PATH]
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
FIRE_STEPS = np.array([0] + [1] * (STEPS - 1), dtype=np.int64)
KW = dict(spread=SPREAD, n_iter=N_ITER, granularity=1.0, boxes=BOXES, h_focus=cov.FullSimulation.H_FOCUS,
          h_max=PARAMS.h_max)


def scenario_starts(E):
    X = np.repeat(START[None], E, axis=0)
    X[1:, :2 * N] += np.rint(np.random.default_rng(7).uniform(-40, 40, size=(E - 1, 2 * N)))
    return X


def fresh(eng):
    ff = cov.DynamicArea.ForestFire(eng, seed=SEED)
    eng.set_params(N, np.full(N, 30 * T_HALF), 1e5, prev_xyR=START, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)
    return ff


def one(eng, ff, x, e, s=S):
    X, obj, st, ms = eng.run_horizon_fire(x, FIRE_STEPS, ff.wind_speed, ff.wind_direction, ff.prob_spread,
                                          ff.seed + e, ff.t + 1, S=s, seed=SEED + e * STEPS * s, **KW)
    return (X, obj, st, eng.fire_state()), float(ms.sum())


def sequential(eng, X0):
    out, ms, busy = [], 0.0, 0.0
    for e in range(X0.shape[0]):
        ff = fresh(eng)
        t0 = time.perf_counter()
        r, m = one(eng, ff, X0[e], e)
        busy += time.perf_counter() - t0
        out.append(r)
        ms += m
    return out, ms, busy


def threaded(engs, ffs, X0):
    E, G = X0.shape[0], len(engs)
    out = [None] * E

    def work(k):
        for i, e in enumerate(range(k, E, G)):
            ff = ffs[k] if i == 0 else fresh(engs[k])
            out[e], _ = one(engs[k], ff, X0[e], e)

    th = [threading.Thread(target=work, args=(k,)) for k in range(G)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    return out, None, None


def ensemble(eng, ff, X0):
    X, obj, st, ms, states = ff.run_horizon_ensemble(X0, FIRE_STEPS, S=S, seed=SEED, want_states=True, **KW)
    return [(X[e], obj[e], {k: v[e] for k, v in st.items()}, states[e]) for e in range(X0.shape[0])], \
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
               all(np.array_equal(x[2][k], y[2][k]) for k in x[2]) and np.array_equal(x[3], y[3])
               for x, y in zip(a, b))


def single_rows():
    """cov_run_horizon_fire at S = 1 and 148 from the base swarm, and 100 cov_fire_step calls on a fresh fire."""
    rows = {}
    with cov.CoverageEngine(0) as eng:
        for s in (1, 148):
            def run():
                ff = fresh(eng)
                t0 = time.perf_counter()
                _, m = one(eng, ff, START, 0, s)
                return None, m, time.perf_counter() - t0
            rows[f"cov_run_horizon_fire S={s}"], _ = measure(run)

        def steps():
            ff = fresh(eng)
            t0 = time.perf_counter()
            for _ in range(100):
                ff.step()
            return None, None, time.perf_counter() - t0
        rows["100 x cov_fire_step"], _ = measure(steps)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r8_horizon_fire_ensemble_rate.json"))
    ap.add_argument("--baseline-tree", default=None, help="another built checkout for the single-scenario rows")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of this build and the baseline build")
    ap.add_argument("--single-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--sizes", default="1,148,1024")
    args = ap.parse_args()
    if args.single_only:  # one build's single-scenario rows, in a process of its own
        print(json.dumps(single_rows()))
        return
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown", "config": "ForestFire 100 x 100 at 5 m (seed 3), N = 5",
           "T": STEPS, "S": S, "N_iter": N_ITER, "spread_m": SPREAD, "seed": SEED, "fire_seed_stride": 1,
           "fire_steps": "0, then 1 per timestep",
           "how": f"host clock, median of {REPEATS} after a warm-up; sequential: only the calls are timed, the fire, "
                  "store and parameters are restored before each outside the clock; threads: handles prepared before "
                  "the clock, restores between a thread's later scenarios inside it", "runs": {}}
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
        for E in [int(v) for v in args.sizes.split(",")]:
            X0 = scenario_starts(E)
            G = min(E, 148)
            ffs = [None] * G

            def prep_threads():
                for k in range(G):
                    ffs[k] = fresh(engs[k])
            r_seq, res_seq = measure(lambda: sequential(eng, X0))
            r_thr, res_thr = measure(lambda: threaded(engs[:G], ffs, X0), prepare=prep_threads)
            ff = fresh(eng)
            r_ens, res_ens = measure(lambda: ensemble(eng, ff, X0))
            r_ens["same_bits_as_sequential"] = same(res_ens, res_seq)
            r_thr["same_bits_as_sequential"] = same(res_thr, res_seq)
            row = {"sequential cov_run_horizon_fire": r_seq, f"threads ({G} handles)": r_thr,
                   "cov_run_horizon_fire_ensemble": r_ens,
                   "entries_appended_mean": float(np.mean([r[2]["appended"].sum() for r in res_ens])),
                   "entries_removed_mean": float(np.mean([r[2]["removed"].sum() for r in res_ens])),
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
