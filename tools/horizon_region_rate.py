"""The receding horizon on the grid-free static objective: config 1 (500 m domain, N = 5, T = 40, N_iter 100), from an
empty covered set.

  device       one cov_run_horizon_region call (S = 1 and 148), and the device time per timestep of its kernels
               (the covered set's step with the arcs, the solves, the rest) from torch.profiler in a profiled call
               after the timed ones
  replay       the same horizon from single calls (the test suite's replay: cov_set_region, the r_max rule,
               cov_set_params, cov_mads_solve_batch_region, the argmin, cov_eval_region_batch), without the replay's
               NumPy arc count
  host loop    FullSimulation.run_simulation(objective="region") (the host MADS loop of the reference, S = 1)

The device and replay horizons are checked to be the same bits in the same run.  Wall times from the host clock around
whole horizons (median of 5 after a warm-up; the host loop once).

    python tools/horizon_region_rate.py [--out profiles/r11_horizon_region_rate.json]
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
import test_horizon_region as thr  # noqa: E402

T_HALF = cov.TAN_HALF_FOV_DEFAULT
N, STEPS, N_ITER, SEED, SPREAD, REPEATS = 5, 40, 100, 3, 3.0, 5
PARAMS = cov.FullSimulation.SimulationParameters(N_iter=N_ITER, seed=SEED)
BOXES = cov.FullSimulation._boxes(PARAMS)
START = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T_HALF, 250.0, 250.0)
R0 = np.full(N, PARAMS.h_max * T_HALF)
KW = dict(spread=SPREAD, n_iter=N_ITER, granularity=1.0, seed=SEED, boxes=BOXES, h_focus=cov.FullSimulation.H_FOCUS,
          h_max=PARAMS.h_max)


def fresh(eng):
    eng.set_region(*thr.DOMAIN, None)
    eng.set_params(N, R0, 1e5, prev_xyR=START, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)


def median_ms(fn, reset):
    reset()
    fn()  # warm-up
    ts = []
    for _ in range(REPEATS):
        reset()
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_horizon_region_rate.json"))
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "config": dict(N=N, T=STEPS, N_iter=N_ITER, domain=thr.DOMAIN, repeats=REPEATS), "runs": {}}
    dev, ref = cov.CoverageEngine(0), cov.CoverageEngine(0)
    arcs_only = thr.arc_count  # the replay's restated arc count stays outside the clock
    thr.arc_count = lambda C, domain=thr.DOMAIN: 0
    try:
        for S in (1, 148):
            out = {}

            def run_dev():
                out["dev"] = dev.run_horizon_region(START, STEPS, S=S, **KW)

            def setp(r, prev):
                ref.set_params(N, r, 1e5, prev_xyR=prev, d_lim=PARAMS.d_lim, tan_half_fov=T_HALF)

            def run_ref():
                out["ref"] = thr.replay(cov, ref, np.zeros((0, 3)), START, STEPS, S, SPREAD, N_ITER, 1.0, SEED, BOXES,
                                        KW["h_focus"], KW["h_max"], R0, setp)

            d_ms, d_all = median_ms(run_dev, lambda: fresh(dev))
            r_ms, r_all = median_ms(run_ref, lambda: fresh(ref))
            X, obj, st, step_ms = out["dev"]
            Xr, objr, str_, _, _, failed = out["ref"]
            same = (failed is None and np.array_equal(X.view(np.uint64), Xr.view(np.uint64)) and
                    np.array_equal(obj.view(np.uint64), objr.view(np.uint64)) and
                    all(np.array_equal(st[k], str_[:, q]) for q, k in enumerate(("winner", "evaluations", "feasible"))))
            res["runs"][f"S{S}"] = dict(device_ms=d_ms, device_all_ms=d_all, replay_ms=r_ms, replay_all_ms=r_all,
                                        speedup_vs_replay=r_ms / d_ms, same_bits=bool(same),
                                        step_ms_sum=float(np.sum(step_ms)), step_ms_first=float(step_ms[0]),
                                        step_ms_last=float(step_ms[-1]), arcs_last=int(st["arcs"][-1]))
            print(f"S={S}: device {d_ms:.1f} ms, replay {r_ms:.1f} ms, same bits {same}", flush=True)
        thr.arc_count = arcs_only
        res["split_ms_per_timestep"] = split()
        cells = cov.CellFunctions.initialise_POI(cov.CellFunctions.Cells(), "static")
        t0 = time.perf_counter()
        cov.FullSimulation.run_simulation(cells, START, cov.TDM_Constraints.cons1, [], N, R0.copy(), PARAMS,
                                          Nt_sim=STEPS, objective="region")
        res["host_loop_ms"] = (time.perf_counter() - t0) * 1e3
        cells.close()
        print(f"host loop {res['host_loop_ms']:.1f} ms", flush=True)
    finally:
        dev.close()
        ref.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


def split():
    """Device time per timestep of each kernel of one horizon (S = 1 and 148), from torch.profiler's CUDA activities
    in a profiled call after the timed ones: the arcs step (cover_arcs_kernel) against the solves (cover_solve_kernel)
    and the rest."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    out = {}
    eng = cov.CoverageEngine(0)
    try:
        for S in (1, 148):
            fresh(eng)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                eng.run_horizon_region(START, STEPS, S=S, **KW)
            per = {}
            for e in prof.events():
                if e.device_type.name == "CUDA" and "_kernel" in e.name:
                    key = next((k for k in ("cover_arcs", "cover_solve", "cover_eval", "horizon_start",
                                            "horizon_commit") if k in e.name), e.name)
                    per[key] = per.get(key, 0.0) + e.device_time / 1e3 / STEPS  # us -> ms per timestep
            out[f"S{S}"] = per
            print(f"split S={S}: " + ", ".join(f"{k} {v:.3f} ms" for k, v in per.items()), flush=True)
    finally:
        eng.close()
    return out


if __name__ == "__main__":
    main()
