"""Multi-start MADS on the device: one cov_mads_solve_batch launch for S solves against S sequential cov_mads_solve
calls and against mads.optimize_multistart (the Python lockstep driver, one evaluation launch per iteration).

Two workloads, N = 5 UAVs, N_iter = 100, granularity 1, cons3 (10 m from the starting swarm) fused:
  static   config 1: createPOI on 100 x 100 cells of 5 m, rmvCoveredPOI with the starting swarm
  dynamic  the first 30 rows of the fire list (multiplicities: two bit planes) with the high-interest class of weight
           (30 tan 50 deg)^2 pi on 240 < x < 300 (not dyadic: the list-order Float64 sum)
Starts: allocate_even_circles(15, 5, 10 tan 50 deg, centre) plus seeded integer perturbations of the centres.
Timing: host clock around the synchronous call after one warm-up call, repeated until at least 0.5 s is timed.
The direction streams of the three methods differ, so their objectives are compared as distributions (median, best).

    python tools/mads_batch_rate.py [--out profiles/r3_mads_batch.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import coverage_b200 as cov  # noqa: E402

T = cov.TAN_HALF_FOV_DEFAULT
N, N_ITER, GRAN = 5, 100, 1.0
SIZES = (1, 8, 148, 1024)


class _Objective:
    """obj.batch for mads.optimize_multistart on an engine whose parameters already fuse the constraints."""

    def __init__(self, eng):
        self.eng = eng

    def batch(self, X, want_feasible=False):
        r = self.eng.eval_batch(X, want_count=False, want_feasible=True)
        return (r["obj"], r["feasible"].astype(bool)) if want_feasible else r["obj"]


def timed(fn, min_s=0.5):
    fn()  # warm-up
    reps, t0 = 0, time.perf_counter()
    while True:
        out = fn()
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= min_s:
            return dt / reps, reps, out


def summary(obj):
    f = np.asarray(obj, dtype=np.float64)
    f = f[np.isfinite(f)]
    return {"feasible": int(f.size), "median_objective": float(np.median(f)) if f.size else None,
            "best_objective": float(f.min()) if f.size else None}


def setup(eng, kind):
    if kind == "static":
        centre = (250.0, 250.0)
        eng.set_grid_full(100, 100, 5.0, 5.0)
    else:
        centre = (250.0, 330.0)
        rows = cov.fire_io.load_fire_rows_npz(os.path.join(os.path.dirname(__file__), "..", "tests", "golden",
                                                           "fire_rows.npz"))
        pts = np.concatenate(rows[:30]).copy()
        hi = (pts[:, 0] > 240) & (pts[:, 0] < 300)
        pts[hi, 2] = pts[hi, 3] = (30 * T) ** 2 * math.pi
        eng.set_points(pts, 100, 100, 5.0, 5.0)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, *centre)
    eng.set_params(N, np.full(N, 30 * T))
    eng.remove_covered(x0)
    eng.set_params(N, np.full(N, 30 * T), prev_xyR=x0, d_lim=10.0, tan_half_fov=T)
    return x0


def run(kind):
    eng = cov.CoverageEngine(0)
    x0 = setup(eng, kind)
    info = eng.grid_info()
    rng = np.random.default_rng(2026)
    Xall = np.repeat(x0[None, :], max(SIZES), axis=0)
    Xall[:, :2 * N] += np.rint(rng.normal(0.0, 3.0, (max(SIZES), 2 * N)))
    res = {"store": {k: info[k] for k in ("n_entries", "n_planes", "n_classes", "area_exact")}, "by_S": {}}
    for S in SIZES:
        X0 = Xall[:S]
        row = {}
        t, reps, (X, obj, st) = timed(lambda: eng.mads_solve_batch(X0, N_ITER, GRAN, seed=1))
        ev = int(st["evaluations"].sum())
        row["batch"] = {"wall_ms": t * 1e3, "reps": reps, "solves_per_s": S / t, "evaluations_per_s": ev / t,
                        "mean_iterations": float(st["iterations"].mean()), **summary(obj)}

        def sequential():
            out = [eng.mads_solve(X0[k], N_ITER, GRAN, seed=1 + k) for k in range(S)]
            return np.array([o[1] for o in out]), sum(o[2]["evaluations"] for o in out)
        t, reps, (obj, ev) = timed(sequential)
        row["sequential_mads_solve"] = {"wall_ms": t * 1e3, "reps": reps, "solves_per_s": S / t,
                                        "evaluations_per_s": ev / t, **summary(obj)}
        if S <= 148:
            def lockstep():
                _, o, _, s = cov.mads.optimize_multistart(X0, _Objective(eng), [], [], N_ITER, granularity=GRAN,
                                                          seed=1, return_stats=True)
                return o, s["evaluations"]
            t, reps, (obj, ev) = timed(lockstep)
            row["optimize_multistart_python"] = {"wall_ms": t * 1e3, "reps": reps, "solves_per_s": S / t,
                                                 "evaluations_per_s": ev / t, **summary(obj)}
        row["speedup_vs_sequential"] = row["sequential_mads_solve"]["wall_ms"] / row["batch"]["wall_ms"]
        res["by_S"][str(S)] = row
        print(kind, S, json.dumps(row), flush=True)
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r3_mads_batch.json"))
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"gpu": gpu[0] if gpu else "unknown", "N": N, "N_iter": N_ITER, "granularity": GRAN,
           "how": "host clock around synchronous calls after a warm-up call, >= 0.5 s timed per entry",
           "static": run("static"), "dynamic": run("dynamic")}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
