"""Rates of the grid-free static objective against the grid objective on the same swarms.

  eval     cov_eval_region_batch on 1 M candidates (synth.random_candidates: x, y ~ U(0, 500), h ~ U(5, 30),
           R = h tan 50 deg) at N = 5 and 64 with M = 0 and 200 covered discs; kernel time from CUDA events around the
           evaluation kernel(s) (cov_last_kernel_ms: the candidates are device-resident while it runs), and the wall
           time of the whole synchronous call (H2D of the candidates and D2H of the results included).
  grid     cov_eval_batch_device on the same candidates already on the device (cov_last_kernel_ms), config 1's
           createPOI at 5 m and the finest lattice the grid path accepts (32768 x 32768: 2^-6 * 500 m cells), the
           starting swarm removed; at the finest lattice on 2^16 candidates (a longer run is not needed for a rate).
  mads     148 and 1024 solves of cov_mads_solve_batch_region on config 1 (covered set: 195 discs of earlier rings
           and the starting swarm, cons3 at 10 m from it, N_iter 100, granularity 1), host clock around the synchronous
           call after a warm-up; cov_mads_solve_batch on config 1's grid for comparison.
The card's name and power limit are read in the same run.  Writes JSON.

    python tools/region_rate.py [--out profiles/r4_region_rate.json]
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
DOMAIN = (0.0, 0.0, 500.0, 500.0)


def covered_set(rng, M):
    out = []
    while len(out) < M:
        cx, cy, R = rng.uniform(0, 500), rng.uniform(0, 500), rng.uniform(5, 35)
        for i in range(5):
            a = 2 * math.pi * i / 5
            out.append([cx + 15 * math.cos(a), cy + 15 * math.sin(a), R])
    return np.array(out[:M]).reshape(-1, 3)


def median_of(fn, reps=3):
    fn()  # warm-up
    return float(np.median([fn() for _ in range(reps)]))


def eval_rates(eng, B):
    out = {}
    rng = np.random.default_rng(1)
    for N in (5, 64):
        X = cov.synth.random_candidates(B, N, seed=N)
        eng.set_params(N, np.full(N, 30 * T))
        for M in (0, 200):
            eng.set_region(*DOMAIN, covered_set(rng, M))

            def kernel():
                eng.eval_region_batch(X, want_area=False, want_feasible=False)
                return eng.last_kernel_ms()

            def wall():
                t0 = time.perf_counter()
                eng.eval_region_batch(X, want_area=False, want_feasible=False)
                return (time.perf_counter() - t0) * 1e3

            k, w = median_of(kernel), median_of(wall)
            out[f"N{N}_M{M}"] = {"B": B, "kernel_ms": k, "evals_per_s_kernel": B / k * 1e3, "call_ms": w,
                                 "evals_per_s_call": B / w * 1e3}
            print(N, M, out[f"N{N}_M{M}"], flush=True)
    return out


def grid_rates(eng, B):
    out = {}
    N = 5
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    for n, Bn in ((100, B), (32768, 1 << 16)):
        eng.set_grid_full(n, n, 500.0 / n, 500.0 / n)
        eng.set_params(N, np.full(N, 30 * T))
        eng.remove_covered(x0)
        X = cov.synth.random_candidates(Bn, N, seed=N)
        dX, dO = eng.device_alloc(X.nbytes), eng.device_alloc(Bn * 8)
        eng.memcpy_h2d(dX, X)
        eng.sync()

        def kernel():
            eng.eval_batch_device(dX, Bn, dO)
            eng.sync()
            return eng.last_kernel_ms()

        k = median_of(kernel)
        out[f"grid_{n}x{n}_N5"] = {"B": Bn, "dx_m": 500.0 / n, "kernel_ms": k, "evals_per_s_kernel": Bn / k * 1e3}
        print(n, out[f"grid_{n}x{n}_N5"], flush=True)
        eng.device_free(dX)
        eng.device_free(dO)
    return out


def mads_rates(eng):
    out = {}
    N = 5
    rng = np.random.default_rng(5)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    C3 = np.concatenate([covered_set(rng, 195), x0.reshape(3, N).T])
    for S in (148, 1024):
        X0 = np.repeat(x0[None, :], S, axis=0)
        X0[:, :2 * N] += np.rint(rng.normal(0, 3.0, (S, 2 * N)))
        for kind in ("region", "grid_100x100"):
            if kind == "region":
                eng.set_params(N, np.full(N, 30 * T), prev_xyR=x0, d_lim=10.0, tan_half_fov=T)
                eng.set_region(*DOMAIN, C3)
                solve = lambda: eng.mads_solve_batch_region(X0, 100, 1.0, 7)  # noqa: E731
            else:
                eng.set_grid_full(100, 100, 5.0, 5.0)
                eng.set_params(N, np.full(N, 30 * T))
                eng.remove_covered(x0)
                eng.set_params(N, np.full(N, 30 * T), prev_xyR=x0, d_lim=10.0, tan_half_fov=T)
                solve = lambda: eng.mads_solve_batch(X0, 100, 1.0, 7)  # noqa: E731
            res = {}

            def run():
                t0 = time.perf_counter()
                res["r"] = solve()
                return (time.perf_counter() - t0) * 1e3

            ms = median_of(run)
            X, obj, st = res["r"]
            ev = int(st["evaluations"].sum())
            out[f"S{S}_{kind}"] = {"wall_ms": ms, "solves_per_s": S / ms * 1e3, "evaluations": ev,
                                   "evaluations_per_s": ev / ms * 1e3, "mean_iterations": float(st["iterations"].mean()),
                                   "feasible": int(np.isfinite(obj).sum()),
                                   "median_objective": float(np.median(obj[np.isfinite(obj)]))}
            print(S, kind, out[f"S{S}_{kind}"], flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r4_region_rate.json"))
    ap.add_argument("--batch", type=int, default=1 << 20)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    with cov.CoverageEngine(0) as eng:
        res = {"gpu": gpu, "how": __doc__.split("\n\n")[1], "eval": eval_rates(eng, a.batch),
               "grid": grid_rates(eng, a.batch), "mads": mads_rates(eng)}
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
