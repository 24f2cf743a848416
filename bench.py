#!/usr/bin/env python
"""bench.py -- coverage-objective throughput of libcoverage_cuda on BASELINE.json's workload.

Workload (config.workload): BASELINE.json configs[1] -- 5 UAVs x 1 M random candidates per launch on a
256 x 256 synthetic fire grid, per GPU (weak scaling: every rank evaluates its own candidates).
One "step" = LAUNCHES (default 40) back-to-back passes of the hot path, each over its own batch of 1 M
candidates (40 distinct device-resident sets, 4.8 GB), so that 20 steps time > 0.5 s of GPU work.

  value      evals/s with the candidates already resident in HBM (cov_eval_batch_device), CUDA events on
             the launching stream, max over ranks.
  e2e        evals/s through the reference-facing call cov_eval_batch with pinned HOST buffers: the
             host->device copy of the candidates and the device->host copy of objective / count /
             feasibility are inside the timed region.  With several ranks every call also ends with
             the path's only exchange (SURVEY.md 8e): the 16-byte (min objective, global index) pair
             of the rank's poll winner, all-gathered over NCCL (cov_eval_batch_best + all_gather).
  e2e_pageable  the same call with plain NumPy (pageable) buffers -- what a Julia `Vector` is.
  e2e_gather    (ranks > 1) a pipelined H2D -> kernel -> NCCL all_gather_into_tensor of the objective
             vectors -> D2H of the gathered vector: the "gather the objective vector" variant of 8e.
  roofline   the bound that matters: instruction ISSUE.  achieved = executed warp instructions per
             candidate (ncu capture of exactly this kernel instantiation on this workload, profiles/
             r2_issue.json, re-measured whenever csrc/ changes) x candidates / live event-timed kernel
             time; peak = 148 SMs x 4 schedulers x the SM clock sampled during the run.
  roofline_hbm  the HBM view the contract also asks for (algorithmic bytes / kernel time / measured peak).
  extra_workloads  short runs of the other BASELINE configs: C3 (50 UAVs, 1024^2, cons8), C4 (200 UAVs,
             4096^2, cons8; candidate-sharded over the ranks = strong scaling) and the C1 poll (30-point
             MADS poll latency and ms per native MADS solve), each with a bit-exact oracle check.
  cpu_baseline  oracle/coverage_oracle.c (a literal C port of the reference's Julia arithmetic;
             Julia itself is not installed) on the host cores, bounded sample, rank 0 / N=1.

`--impl reference` times that CPU port alone, all host threads, on the same workload; it never loads
libcoverage_cuda (synth.py is imported by file path).

`--dump-outputs DIR` writes what the last device-resident launch of the last timed step returned (rank 0):
obj.npy and count.npy (float64) and feasible.npy (float32), one row per candidate.  The candidates come from
the seeded device generator, so the same arguments give the same inputs on every run and two builds can be
compared output for output.  Above 64 MB in all a fixed, seeded sample of the rows is written, with their
row numbers in index.npy.
"""
from __future__ import annotations

import argparse
import hashlib
import importlib.util
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = os.path.join(ROOT, "maximumareacoverageoptimization.jl_b200")

WORKLOADS = {
    "c2": dict(n=5, grid=256, batch=1_000_000, sep=0.0, launches=40,
               name="C2: 5 UAVs x 1M random candidates/launch/GPU, 256x256 synthetic fire grid (BASELINE.json configs[1])"),
    "c3": dict(n=50, grid=1024, batch=65_536, sep=15.0, launches=4,
               name="C3 (reduced batch): 50 UAVs x 64K candidates/launch, 1024x1024 fire grid, cons8 separation (configs[2])"),
    "c4": dict(n=200, grid=4096, batch=8_192, sep=15.0, launches=2,
               name="C4 (reduced batch): 200 UAVs x 8K candidates/launch, 4096x4096 fire grid, cons8 separation (configs[3])"),
    "c1": dict(n=5, grid=100, batch=1_000_000, sep=0.0, launches=40,
               name="C1 grid (100x100, dx=5, dense createPOI) with 1M random candidates/launch/GPU"),
}
HOST_SETS = 8  # distinct pinned host candidate sets the e2e launches rotate over
METRIC = "coverage_objective_evals_per_sec"
UNIT = "evals/s"
ISSUE_PROFILE = os.path.join(ROOT, "profiles", "r2_issue.json")


def load_synth():
    """synth.py by file path: NumPy only, does not import the package (and so never dlopens libcoverage_cuda)."""
    spec = importlib.util.spec_from_file_location("cov_synth_standalone", os.path.join(PKG, "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def source_sha() -> str:
    """Hash of the CUDA sources: an ncu capture is only evidence for the code it was taken from."""
    h = hashlib.sha256()
    d = os.path.join(PKG, "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(d, f), "rb") as fh:
                h.update(f.encode() + b"\0" + fh.read())
    return h.hexdigest()[:16]


def kernel_key(li: dict) -> str:
    """Name of the template instantiation a launch ran (cov_last_launch)."""
    if li["kernel"] == 1:
        return f"span_small_kernel<{li['multi']},{li['chunk']},{li['max_warps']}>"
    if li["kernel"] == 4:
        return f"span_cta_kernel<{li['multi']},{li['plane_mode']},{li['chunk']}>"
    return {2: "brute_kernel", 3: "exact_kernel"}.get(li["kernel"], f"kernel{li['kernel']}")


def load_issue_profile():
    if not os.path.exists(ISSUE_PROFILE):
        return {}
    with open(ISSUE_PROFILE) as f:
        return json.load(f)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback", 1965.0


def issue_view(profile: dict, workload: str, key: str, batch: int, kernel_ms: float, sm_mhz: float, strict: bool):
    """Issue-slot roofline of one kernel: warp instructions per candidate (ncu) x candidates / live time over
    148 SMs x 4 schedulers x clock.  strict: the named workload at its named batch MUST have a profile."""
    ent = profile.get("kernels", {}).get(f"{workload}|{key}")
    if ent is None:
        if strict and not os.environ.get("COV_BENCH_ALLOW_MISSING_PROFILE"):  # (development: before the first capture)
            raise SystemExit(f"bench.py: no ncu issue profile for '{workload}|{key}' in {ISSUE_PROFILE}; "
                             f"re-run tools/issue_profile.py (see profiles/README.md) before benchmarking")
        return {"bound": "issue", "achieved": None, "peak": 148 * 4 * sm_mhz * 1e6, "unit": "warp-instr/s", "frac": None,
                "kernel": key, "note": "no ncu capture for this instantiation (non-default batch / workload)"}
    wipc = float(ent["warp_instr_per_candidate"])
    achieved = wipc * batch / (kernel_ms * 1e-3)
    peak = 148 * 4 * sm_mhz * 1e6
    out = {"bound": "issue", "achieved": achieved, "peak": peak, "unit": "warp-instr/s", "frac": achieved / peak,
           "kernel": key, "kernel_ms": kernel_ms, "warp_instr_per_candidate": wipc, "sm_mhz": sm_mhz,
           "traffic": ent.get("dram_bytes_per_launch"), "profile": os.path.relpath(ISSUE_PROFILE, ROOT),
           "profile_ncu_issue_active_pct": ent.get("issue_active_pct"),
           "peak_source": "148 SMs x 4 issue slots x SM clock sampled by nvidia-smi during the timed region"}
    if profile.get("source_sha") != source_sha():
        out["profile_stale"] = True  # csrc/ changed after the capture: the instruction count may be off
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            inside = t0 <= ts <= t1 + 0.05
            try:
                if inside:
                    sm.append(float(f[1]))
                    power.append(float(f[3]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            if inside:
                for name, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        note = None
        if not sm:  # region shorter than the sampling period: use every sample we have
            note = "no sample inside the timed region; all samples used"
            for ts, line in self.lines:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1]))
                except (ValueError, IndexError):
                    pass
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
               "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}
        if note:
            out["note"] = note
        return out


def bind_to_gpu_numa_node(local: int):
    """Pin this rank to the CPUs next to its GPU before any pinned host memory is allocated (first touch
    then places the staging pages on the GPU's NUMA node). Best effort: returns a note for the JSON line."""
    try:
        import torch
        prop = torch.cuda.get_device_properties(local)
        bus = f"{getattr(prop, 'pci_domain_id', 0):04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bus}/local_cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if use and use != allowed:
            os.sched_setaffinity(0, use)
            return f"bound to {len(use)} CPUs local to {bus}"
        return f"no narrower local CPU set for {bus} ({len(allowed)} CPUs allowed)"
    except Exception as e:  # noqa: BLE001  (sysfs layout, permissions, torch version)
        return f"not bound ({type(e).__name__})"


def make_workload(synth, wl):
    n = wl["grid"]
    d = 5.0 if n == 100 else 500.0 / n
    bits, n_fire = synth.fire_grid(n, dense=(n == 100))
    r_max = np.full(wl["n"], 30.0 * synth.TAN_HALF_FOV_DEFAULT)
    return bits, n_fire, d, r_max


def cpu_port_rate(synth, wl, bits, d, r_max, seconds: float, threads: int = 0, seed: int = 12345):
    """evals/s of the CPU port (oracle/coverage_oracle.c) on a bounded sample of the workload."""
    from oracle import c_oracle
    N, sep = wl["n"], wl["sep"]
    pts = synth.points_from_bits(bits, wl["grid"], d, d)
    nthr = c_oracle.num_threads() if threads <= 0 else threads
    X = synth.random_candidates(max(2048, 128 * nthr), N, seed=seed)
    c_oracle.eval_batch(X[:256], N, r_max, pts, sep_min=sep, threads=threads)  # thread start-up, page-in
    t = time.perf_counter()
    c_oracle.eval_batch(X, N, r_max, pts, sep_min=sep, threads=threads)
    rate = len(X) / (time.perf_counter() - t)
    n = int(max(len(X), min(rate * seconds, 4_000_000)))
    X = synth.random_candidates(n, N, seed=seed + 1)
    t = time.perf_counter()
    out = c_oracle.eval_batch(X, N, r_max, pts, sep_min=sep, threads=threads)
    dt = time.perf_counter() - t
    return n / dt, nthr, n, dt, out, X, pts


def run_reference(args, wl):
    """The reference arm: the CPU port of the reference's objective on all host threads.  Loads
    oracle/libcoverage_oracle.so only -- never the product library."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    synth = load_synth()
    from oracle import c_oracle
    N, sep = wl["n"], wl["sep"]
    bits, n_fire, d, r_max = make_workload(synth, wl)
    pts = synth.points_from_bits(bits, wl["grid"], d, d)
    nthr = c_oracle.num_threads()
    # one step = a bounded sample of the workload: sized for ~2 s of CPU work per step
    probe = synth.random_candidates(max(256, 64 * nthr), N, seed=99)
    c_oracle.eval_batch(probe, N, r_max, pts, sep_min=sep, threads=0)  # thread start-up, page-in
    t = time.perf_counter()
    c_oracle.eval_batch(probe, N, r_max, pts, sep_min=sep, threads=0)
    rate = len(probe) / (time.perf_counter() - t)
    per_launch = wl["batch"] * wl["launches"]
    budget_s = 100.0 / max(args.steps + args.warmup, 1)  # the whole run should end within ~2 minutes
    per_step = int(max(256, min(rate * min(2.0, budget_s), per_launch)))
    X = synth.random_candidates(per_step, N, seed=1)
    for _ in range(args.warmup):
        c_oracle.eval_batch(X, N, r_max, pts, sep_min=sep, threads=0)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        c_oracle.eval_batch(X, N, r_max, pts, sep_min=sep, threads=0)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = f"{per_step} of the step's {per_launch} candidates per step, {args.steps} steps"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"], "uavs": N, "grid": f"{wl['grid']}x{wl['grid']}", "fire_entries": n_fire,
                   "candidates_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthr, "kind": "port", "sample": sample,
                         "note": "C port of the reference's Julia objective (Julia is not installed); "
                                 "pthreads over candidates"},
        "tests_per_sec": value * n_fire * N,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))
    return 0


# ------------------------------------------------------------------------------------------------
class Ctx:
    """What every measurement needs: torch, dist, the package, rank layout, the stream."""


def barrier(c):
    if c.world > 1:
        c.dist.barrier()
    c.torch.cuda.synchronize()


def max_over_ranks(c, values):
    t = c.torch.tensor(values, dtype=c.torch.float64, device=f"cuda:{c.local}")
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    return [float(v) for v in t.tolist()]


def device_resident(c, eng, wl, B, launches, steps, warmup, n_sets, seed0, sampler=None):
    """K steps of `launches` back-to-back cov_eval_batch_device calls over distinct resident candidate sets.
    Returns (ms for the K steps [events, max over ranks], average kernel ms [library events], launches, key)."""
    torch = c.torch
    N = wl["n"]
    row = 3 * N * 8
    dX = [eng.device_alloc(B * row) for _ in range(n_sets)]
    d_obj, d_cnt, d_fe = eng.device_alloc(B * 8), eng.device_alloc(B * 8), eng.device_alloc(B)
    for k in range(n_sets):
        eng.generate_candidates(dX[k], B, N, seed=seed0, first_index=k * B)
    eng.sync()

    def step(s):
        for l in range(launches):
            eng.eval_batch_device(dX[(s * launches + l) % n_sets], B, d_obj, d_cnt, d_fe)

    with torch.cuda.stream(c.stream):
        for s in range(warmup):
            step(s)
        barrier(c)
        ms0, l0 = eng.kernel_time_total()
        launches0 = eng.launch_count()
        if sampler is not None:
            sampler.start()
            time.sleep(0.2)
        barrier(c)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall0 = time.perf_counter()
        e0.record(c.stream)
        for s in range(steps):
            step(s)
        e1.record(c.stream)
        barrier(c)
        t_wall1 = time.perf_counter()
        dev_ms = e0.elapsed_time(e1)
        ms1, l1 = eng.kernel_time_total()
        n_launch = eng.launch_count() - launches0
    kernel_ms = (ms1 - ms0) / max(l1 - l0, 1)
    key = kernel_key(eng.last_launch())
    # every launch writes the same output buffers: they hold the last launch of the last step
    obj = np.empty(B)
    cnt = np.empty(B, dtype=np.int64)
    fe = np.empty(B, dtype=np.uint8)
    eng.memcpy_d2h(obj, d_obj)
    eng.memcpy_d2h(cnt, d_cnt)
    eng.memcpy_d2h(fe, d_fe)
    eng.sync()
    for p in dX + [d_obj, d_cnt, d_fe]:
        eng.device_free(p)
    dev_ms, kernel_ms = max_over_ranks(c, [dev_ms, kernel_ms])
    return dict(dev_ms=dev_ms, kernel_ms=kernel_ms, launches=int(n_launch), key=key, wall=(t_wall0, t_wall1),
                count_sum=int(cnt.sum()), obj_finite=bool(np.isfinite(obj).all()),
                outputs={"obj": obj, "count": cnt, "feasible": fe})


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir: str, outputs: dict, seed: int = 0):
    """obj / count as float64 and feasible as float32, <name>.npy each (see the module docstring)."""
    arrays = {"obj": outputs["obj"].astype(np.float64), "count": outputs["count"].astype(np.float64),
              "feasible": outputs["feasible"].astype(np.float32)}
    n = len(arrays["obj"])
    row_bytes = sum(a.itemsize for a in arrays.values())
    budget = DUMP_LIMIT_BYTES - 4096  # room for the .npy headers
    if n * row_bytes > budget:
        keep = budget // (row_bytes + 8)  # + 8: index.npy
        idx = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def h2d_ceiling(c, eng, nbytes=120_000_000, reps=12, sets=4, d2h_bytes=0):
    """What the box can do: every rank copies `nbytes` of pinned host memory to its GPU `reps` times, all ranks
    at once, nothing else running.  The source rotates over `sets` distinct buffers, like the end-to-end run's
    candidate sets, so that the host's last-level cache cannot stand in for its DRAM.  GB/s summed over the ranks
    (max-over-ranks time).
    d2h_bytes > 0: the same with the path's result traffic flowing the other way -- beside copy k+1 a second stream
    copies d2h_bytes (17 B per candidate of copy k) from the device into pinned host memory.  Still H2D GB/s."""
    torch = c.torch
    hosts = [eng.pinned((nbytes // 8,)) for _ in range(sets)]
    for h in hosts:
        h[:] = 1.0
    dev = eng.device_alloc(nbytes)
    back = None
    if d2h_bytes:
        back = (torch.zeros(d2h_bytes, dtype=torch.uint8, device=torch.device("cuda", c.local)),
                torch.empty(d2h_bytes, dtype=torch.uint8, pin_memory=True), torch.cuda.Stream(device=c.local))
    with torch.cuda.stream(c.stream):
        for k in range(sets):
            eng.memcpy_h2d(dev, hosts[k])
        c.torch.cuda.synchronize()
        barrier(c)
        t0 = time.perf_counter()
        for k in range(reps):
            eng.memcpy_h2d(dev, hosts[k % sets])
            if back is not None:
                ev = torch.cuda.Event()
                ev.record(c.stream)
                back[2].wait_event(ev)
                with torch.cuda.stream(back[2]):
                    back[1].copy_(back[0], non_blocking=True)
        c.torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    barrier(c)
    eng.device_free(dev)
    (dt,) = max_over_ranks(c, [dt])
    return c.world * nbytes * reps / dt / 1e9


def e2e_runs(c, eng, cov, wl, B, launches, steps, warmup):
    """The host-facing measurements (wall clock around synchronous calls, barrier + synchronize on both sides)."""
    torch, dist = c.torch, c.dist
    N = wl["n"]
    row = 3 * N * 8
    res = {}
    # pinned host candidate sets, filled from the device generator (distinct per rank and set)
    Xh = [eng.pinned((B, 3 * N)) for _ in range(HOST_SETS)]
    tmp = eng.device_alloc(B * row)
    for k in range(HOST_SETS):
        eng.generate_candidates(tmp, B, N, seed=1000 + c.rank, first_index=k * B)
        eng.memcpy_d2h(Xh[k], tmp)
    eng.sync()
    eng.device_free(tmp)
    out = {"obj": eng.pinned((B,)), "count": eng.pinned((B,), np.int64), "feasible": eng.pinned((B,), np.uint8)}

    from coverage_b200 import distributed as cdist  # (imports torch.distributed: not part of the package's own imports)
    scratch = cdist.exchange_scratch() if c.world > 1 else None
    winners = []

    def call_pinned(k):
        if c.world == 1:
            eng.eval_batch(Xh[k % HOST_SETS], out=out)  # synchronous on return: results are in host memory
            return
        # several ranks: the call also yields this rank's poll winner; the ranks exchange the 16-byte pairs
        r = eng.eval_batch_best(Xh[k % HOST_SETS], barrier=True, out=out)
        bo, bi = r["best"]
        winners.append(cdist.exchange_winner(bo, bi, c.rank * B, scratch)[2])

    def timed(fn):
        for k in range(max(warmup, 1) * 2):
            fn(k)
        barrier(c)
        t0 = time.perf_counter()
        for s in range(steps):
            for l in range(launches):
                fn(s * launches + l)
        barrier(c)
        return (time.perf_counter() - t0) * 1e3

    with torch.cuda.stream(c.stream):
        res["pinned_ms"] = timed(call_pinned)
        if c.world > 1:  # the same call without the winner exchange (what the exchange and its device-side reduction cost)
            res["noexch_ms"] = timed(lambda k: eng.eval_batch(Xh[k % HOST_SETS], out=out))
        # pageable buffers (plain NumPy arrays: what julia/CoverageCUDA.jl's objective_batch passes)
        Xp = [np.array(x) for x in Xh[:4]]
        outp = {"obj": np.empty(B), "count": np.empty(B, dtype=np.int64), "feasible": np.empty(B, dtype=np.uint8)}
        res["pageable_ms"] = timed(lambda k: eng.eval_batch(Xp[k % 4], out=outp))
        del Xp
        # candidates on the MADS mesh (granularity 1.0 on every variable, src/TDM_STATIC_opt.jl:131-137), sent as
        # int16 mesh indices through cov_eval_batch_packed: a quarter of the bytes over PCIe, the same doubles in
        # the kernels.  Same call shape as above (pinned buffers; winner + exchange when there are several ranks).
        synth = cov.synth
        Qh = [eng.pinned((B, 3 * N), np.int16) for _ in range(HOST_SETS)]
        for k in range(HOST_SETS):
            synth.mesh_candidates(B, N, seed=5000 + 97 * c.rank + k, out=Qh[k])

        def call_mesh(k):
            if c.world == 1:
                eng.eval_batch_packed(Qh[k % HOST_SETS], 1.0, out=out)
                return
            r = eng.eval_batch_packed(Qh[k % HOST_SETS], 1.0, best=True, barrier=True, out=out)
            bo, bi = r["best"]
            cdist.exchange_winner(bo, bi, c.rank * B, scratch)

        res["mesh_ms"] = timed(call_mesh)
        # the packed call against cov_eval_batch on the widened matrix (all of one set), bit for bit
        call_mesh(0)
        got = {k: np.array(v) for k, v in out.items()}
        wide = eng.eval_batch(Qh[0].astype(np.float64))
        res["mesh_same"] = float(all(np.array_equal(got[k], wide[k]) for k in ("obj", "count", "feasible")))
        res["mesh_sample"] = (Qh[0][:2048].copy(), got["obj"][:2048].copy(), got["count"][:2048].copy())
        if c.world > 1:
            # gather-the-objective-vector variant: double-buffered H2D (copy stream) -> kernel -> NCCL
            # all_gather_into_tensor of the objective slices -> D2H of the gathered vector (pinned)
            copy_s = torch.cuda.Stream(device=c.local)
            Xt = [torch.from_numpy(x) for x in Xh]
            Xd = [torch.empty((B, 3 * N), dtype=torch.float64, device=f"cuda:{c.local}") for _ in range(2)]
            od = [torch.empty(B, dtype=torch.float64, device=f"cuda:{c.local}") for _ in range(2)]
            gd = [torch.empty(B * c.world, dtype=torch.float64, device=f"cuda:{c.local}") for _ in range(2)]
            gh = torch.from_numpy(eng.pinned((B * c.world,)))
            ev_in = [torch.cuda.Event() for _ in range(2)]
            ev_free = [torch.cuda.Event() for _ in range(2)]

            def gather_step(s):
                for l in range(launches):
                    k = s * launches + l
                    slot = k & 1
                    with torch.cuda.stream(copy_s):
                        copy_s.wait_event(ev_free[slot])
                        Xd[slot].copy_(Xt[k % HOST_SETS], non_blocking=True)
                        ev_in[slot].record(copy_s)
                    c.stream.wait_event(ev_in[slot])
                    eng.eval_batch_device(Xd[slot].data_ptr(), B, od[slot].data_ptr())
                    ev_free[slot].record(c.stream)
                    dist.all_gather_into_tensor(gd[slot], od[slot])
                    gh.copy_(gd[slot], non_blocking=True)
                c.stream.synchronize()

            for s in range(2):
                gather_step(s)
            barrier(c)
            t0 = time.perf_counter()
            for s in range(steps):
                gather_step(s)
            barrier(c)
            res["gather_ms"] = (time.perf_counter() - t0) * 1e3
    sample = res.pop("mesh_sample")
    same = res.pop("mesh_same")
    keys = sorted(res)
    vals = max_over_ranks(c, [res[k] for k in keys])
    res = dict(zip(keys, vals))
    res["winner_exchanges"] = len(winners)
    res["mesh_same"], res["mesh_sample"] = bool(same), sample
    return res


def extra_workload(c, cov, synth, name, profile, sm_mhz, steps=3, warmup=2):
    """A short run of another BASELINE config, candidate-sharded over the ranks (strong scaling), with a
    bit-exact oracle check on a small sample (rank 0)."""
    wl = WORKLOADS[name]
    N = wl["n"]
    bits, n_fire, d, r_max = make_workload(synth, wl)
    eng = cov.CoverageEngine(c.local)
    eng.set_stream(c.stream.cuda_stream)
    eng.set_grid_bits(bits, wl["grid"], wl["grid"], d, d)
    eng.set_params(N, r_max, sep_min=wl["sep"])
    B_total = wl["batch"]
    B = (B_total + c.world - 1) // c.world
    m = device_resident(c, eng, wl, B, wl["launches"], steps, warmup, wl["launches"] + 1, seed0=31 + c.rank)
    total = B * c.world * wl["launches"] * steps
    value = total / (m["dev_ms"] * 1e-3)
    line = {"workload": wl["name"], "uavs": N, "grid": f"{wl['grid']}x{wl['grid']}", "fire_entries": n_fire,
            "candidates_per_launch_per_gpu": B, "launches_per_step": wl["launches"], "steps": steps,
            "scaling": "strong" if c.world > 1 else "n/a", "value": value, "unit": UNIT,
            "tests_per_sec": value * n_fire * N, "kernel": m["key"], "kernel_ms": m["kernel_ms"],
            "roofline": issue_view(profile, name, m["key"], B, m["kernel_ms"], sm_mhz,
                                   strict=(c.world == 1 and B == wl["batch"]))}
    if c.rank == 0:
        from oracle import c_oracle
        ns = {"c3": 256, "c4": 24}.get(name, 2048)
        Xs = synth.random_candidates(ns, N, seed=77)
        pts = synth.points_from_bits(bits, wl["grid"], d, d)
        t = time.perf_counter()
        want = c_oracle.eval_batch(Xs, N, r_max, pts, sep_min=wl["sep"])
        dt = time.perf_counter() - t
        got = eng.eval_batch(Xs)
        line["parity_on_sample"] = bool(np.array_equal(got["count"], want["count"]) and
                                        np.array_equal(got["obj"], want["obj"]) and
                                        np.array_equal(got["feasible"], want["feasible"]))
        line["cpu_port_evals_per_sec"] = ns / dt
        line["parity_sample"] = f"{ns} candidates, counts + Float64 objectives + cons8 flags bit-exact vs the C port"
    eng.close()
    return line


def c1_poll(c, cov, synth, steps=200):
    """BASELINE configs[0]: the reference's own CPU-runnable case.  Latency of one 30-point MADS poll set through
    cov_eval_batch and of one whole native MADS solve (cov_mads_solve, N_iter = 100, granularity 1, cons3 fused)."""
    from oracle import c_oracle
    T = cov.TAN_HALF_FOV_DEFAULT
    N = 5
    eng = cov.CoverageEngine(c.local)
    eng.set_grid_full(100, 100, 5.0, 5.0)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    r_max = np.full(N, 30.0 * T)
    eng.set_params(N, r_max, prev_xyR=x0, d_lim=10.0, tan_half_fov=T)
    rng = np.random.default_rng(5)
    P = np.rint(x0 + rng.normal(0, 3.0, (30, 3 * N)))  # a poll set on the integer mesh around the start point
    pts = c_oracle.createPOI(5.0, 5.0, 100.0, 100.0)
    want = c_oracle.eval_batch(P, N, r_max, pts, pre=x0, d_lim=10.0, tan_half_fov=T)
    got = eng.eval_batch(P)
    ok = bool(np.array_equal(got["obj"], want["obj"]) and np.array_equal(got["count"], want["count"]) and
              np.array_equal(got["feasible"], want["feasible"]))
    for _ in range(20):
        eng.eval_batch(P)
    t = time.perf_counter()
    for _ in range(steps):
        eng.eval_batch(P)
    poll_us = (time.perf_counter() - t) / steps * 1e6
    key = kernel_key(eng.last_launch())
    for s in range(3):
        eng.mads_solve(x0, 100, 1.0, seed=s)
    t = time.perf_counter()
    evals = 0
    n_solves = 20
    for s in range(n_solves):
        x, fo, st = eng.mads_solve(x0, 100, 1.0, seed=100 + s)
        evals += st["evaluations"]
    solve_ms = (time.perf_counter() - t) / n_solves * 1e3
    fo_ref = c_oracle.objective(x, r_max, pts)[0]
    eng.close()
    t = time.perf_counter()
    for _ in range(20):
        c_oracle.eval_batch(P, N, r_max, pts, pre=x0, d_lim=10.0, tan_half_fov=T, threads=1)
    cpu_poll_us = (time.perf_counter() - t) / 20 * 1e6
    return {"workload": "C1: FullSimulation.jl default, 5 UAVs on createPOI(5,5,100,100) (10 000 points), cons3 fused "
                        "(BASELINE.json configs[0])",
            "poll_points": 30, "poll_latency_us": poll_us, "poll_evals_per_sec": 30 / (poll_us * 1e-6), "kernel": key,
            "cpu_port_poll_latency_us_1_thread": cpu_poll_us,
            "mads_solve_ms": solve_ms, "mads_evaluations_per_solve": evals / n_solves,
            "reference_recorded_median_s_per_solve": 0.074,
            "parity_on_sample": ok and fo == fo_ref,
            "parity_sample": "30-point poll set (obj, count, cons3 flag) and the final incumbent's objective vs the C port"}


def main():
    sys.dont_write_bytecode = True  # the tree may be read-only: leave no __pycache__ behind in it
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "span", "brute", "exact"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="candidates per launch per GPU (default: the workload's)")
    ap.add_argument("--launches", type=int, default=0, help="launches per step (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C3 / C4 / C1 sub-runs")
    ap.add_argument("--no-e2e", action="store_true", help="device-resident measurement only (profiling)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed launch's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    wl = dict(WORKLOADS[args.workload])
    named = args.batch in (0, wl["batch"]) and args.kernel == "auto"
    if args.batch > 0:
        wl["batch"] = args.batch
    if args.launches > 0:
        wl["launches"] = args.launches
    if args.impl == "reference":
        return run_reference(args, wl)

    import torch
    import torch.distributed as dist
    import coverage_b200 as cov
    synth = cov.synth

    c = Ctx()
    c.torch, c.dist = torch, dist
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.rank = int(os.environ.get("RANK", "0"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libcoverage_cuda has no CPU fallback")
    torch.cuda.set_device(c.local)
    numa_note = bind_to_gpu_numa_node(c.local) if c.world > 1 else "single rank: not bound"
    if c.world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", c.local))
    B, N, L = wl["batch"], wl["n"], wl["launches"]
    bits, n_fire, d, r_max = make_workload(synth, wl)

    eng = cov.CoverageEngine(c.local)
    c.stream = torch.cuda.Stream(device=c.local)
    eng.set_stream(c.stream.cuda_stream)  # torch's events see the kernels on this stream
    eng.set_grid_bits(bits, wl["grid"], wl["grid"], d, d)
    eng.set_params(N, r_max, sep_min=wl["sep"])
    kid = {"auto": cov.KERNEL_AUTO, "span": cov.KERNEL_SPAN, "brute": cov.KERNEL_BRUTE, "exact": cov.KERNEL_EXACT}[args.kernel]
    eng.set_option(cov.OPT_KERNEL, kid)
    row_bytes = 3 * N * 8

    # ---- device-resident: L distinct sets (> 126 MB L2 between two uses of the same set) ----
    sampler = ClockSampler(c.local) if c.rank == 0 else None
    m = device_resident(c, eng, wl, B, L, args.steps, args.warmup, L, seed0=1 + c.rank, sampler=sampler)
    clocks = sampler.stop(*m["wall"]) if c.rank == 0 else None
    if args.dump_outputs and c.rank == 0:
        dump_outputs(args.dump_outputs, m["outputs"])

    # ---- host-facing ----
    e = None
    ceiling = None
    if not args.no_e2e:
        ceiling = h2d_ceiling(c, eng, nbytes=B * row_bytes)
        ceiling_duplex = h2d_ceiling(c, eng, nbytes=B * row_bytes, d2h_bytes=B * 17)
        e = e2e_runs(c, eng, cov, wl, B, L, args.steps, args.warmup)

    profile = load_issue_profile()
    hbm_peak, peak_kind, sm_max = load_peaks()
    sm_mhz = (clocks or {}).get("sm_mhz") or sm_max
    line = None
    if c.rank == 0:
        per_step = c.world * B * L
        total = per_step * args.steps
        value = total / (m["dev_ms"] * 1e-3)
        bytes_per_eval = 24 * N + 8 + 8 + 1
        tests_per_eval = n_fire * N
        hbm_achieved = B * bytes_per_eval / (m["kernel_ms"] * 1e-3) / 1e9
        issue_peak_lanes = 148 * 4 * 32 * sm_mhz * 1e6
        roof = issue_view(profile, args.workload, m["key"], B, m["kernel_ms"], sm_mhz, strict=named)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": c.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["dev_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["name"], "uavs": N, "grid": f"{wl['grid']}x{wl['grid']}", "fire_entries": n_fire,
                       "candidates_per_launch_per_gpu": B, "launches_per_step": L, "candidates_per_step": per_step,
                       "kernel": args.kernel,
                       "l2": f"every launch of a step reads its own device-resident candidate set: {L} x "
                             f"{B * row_bytes / 1e6:.0f} MB cycle between two uses of a set (> 126 MB L2)",
                       "penalties": "altitude penalty 1e5*sum|R - r_max|" + (f" + cons8 separation {wl['sep']}" if wl["sep"] > 0 else "")},
            "tests_per_sec": value * tests_per_eval,
            "roofline": roof,
            "roofline_hbm": {"bound": "hbm", "achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                             "frac": hbm_achieved / hbm_peak, "peak_source": f"of {peak_kind}",
                             "algorithmic_bytes_per_launch": B * bytes_per_eval, "bytes_per_eval": bytes_per_eval,
                             "note": "not the bound: the grid lives in shared memory, candidates stream at 137 B/eval"},
            "issue": {"algorithmic_tests_per_sec_per_gpu": B * tests_per_eval / (m["kernel_ms"] * 1e-3),
                      "lane_instr_peak_per_sec": issue_peak_lanes,
                      "brute_force_ceiling_tests_per_sec": issue_peak_lanes / 6.0,
                      "frac_of_brute_force_ceiling": B * tests_per_eval / (m["kernel_ms"] * 1e-3) / (issue_peak_lanes / 6.0)},
            "gpu_launches": m["launches"],
            "host_placement": numa_note,
            "clocks": clocks,
            "check": {"count_sum_last_launch": m["count_sum"], "obj_finite": m["obj_finite"]},
        }
        if e is not None:
            calls = args.steps * L
            e2e = total / (e["pinned_ms"] * 1e-3)
            line["e2e"] = {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": B * row_bytes * L,
                           "d2h_bytes_per_step": B * 17 * L, "ms_per_step": e["pinned_ms"] / args.steps,
                           "ms_per_call": e["pinned_ms"] / calls, "calls_per_step": L, "buffers": "pinned (cov_host_alloc)",
                           "exchange": (f"per call: NCCL all_gather of the 16-byte (min, index) pair of {c.world} ranks, "
                                        f"{e['winner_exchanges']} exchanges on rank 0") if c.world > 1 else "single rank: none"}
            line["e2e_pageable"] = {"value": total / (e["pageable_ms"] * 1e-3), "unit": UNIT,
                                    "ms_per_call": e["pageable_ms"] / calls,
                                    "buffers": "pageable NumPy arrays in and out (what a Julia Vector is)"}
            Qs, obj_s, cnt_s = e["mesh_sample"]
            from oracle import c_oracle  # the checker only: 2048 mesh candidates of the timed sets against the C port
            want = c_oracle.eval_batch(Qs.astype(np.float64), N, r_max, synth.points_from_bits(bits, wl["grid"], d, d),
                                       sep_min=wl["sep"])
            line["e2e_mesh"] = {"value": total / (e["mesh_ms"] * 1e-3), "unit": UNIT, "ms_per_call": e["mesh_ms"] / calls,
                                "h2d_bytes_per_step": B * 3 * N * 2 * L, "d2h_bytes_per_step": B * 17 * L,
                                "buffers": "pinned (cov_host_alloc)",
                                "candidates": "uniform on the MADS mesh of the reference (granularity 1.0 on x, y and R, "
                                              "src/TDM_STATIC_opt.jl:131-137), passed as int16 mesh indices to "
                                              "cov_eval_batch_packed and widened to Float64 on the device",
                                "exchange": "as e2e",
                                "parity_on_sample": bool(e["mesh_same"] and np.array_equal(obj_s, want["obj"]) and
                                                         np.array_equal(cnt_s, want["count"])),
                                "parity_sample": "a whole 1M set bit for bit against cov_eval_batch on the widened "
                                                 "Float64 matrix; 2048 of them against the C port"}
            if "noexch_ms" in e:
                line["e2e_no_exchange"] = {"value": total / (e["noexch_ms"] * 1e-3), "unit": UNIT,
                                           "ms_per_call": e["noexch_ms"] / calls,
                                           "note": "cov_eval_batch per rank, no exchange between the ranks (every rank for itself)"}
            if "gather_ms" in e:
                line["e2e_gather"] = {"value": total / (e["gather_ms"] * 1e-3), "unit": UNIT,
                                      "ms_per_call": e["gather_ms"] / calls,
                                      "exchange": "per call: NCCL all_gather_into_tensor of the objective slices "
                                                  f"({B * 8 / 1e6:.0f} MB per rank), gathered vector copied to pinned host memory",
                                      "h2d_bytes_per_step": B * row_bytes * L, "d2h_bytes_per_step": B * 8 * c.world * L}
            line["h2d_ceiling_gbs"] = ceiling
            line["e2e_frac_of_h2d_ceiling"] = e2e * row_bytes / 1e9 / ceiling
            # the same copies with the results' 17 B per candidate going back at the same time (what the path moves)
            line["h2d_ceiling_with_results_gbs"] = ceiling_duplex
            line["e2e_frac_of_ceiling_with_results"] = e2e * row_bytes / 1e9 / ceiling_duplex
    if not args.no_extra and args.workload == "c2":
        extras = [extra_workload(c, cov, synth, name, profile, sm_mhz) for name in ("c3", "c4")]
        if c.rank == 0:
            extras.append(c1_poll(c, cov, synth))
            line["extra_workloads"] = extras
    if c.rank == 0:
        if c.world == 1 and not args.no_cpu_baseline:
            rate, nthr, n, dt, ref, Xc, pts = cpu_port_rate(synth, wl, bits, d, r_max, args.cpu_seconds)
            got = eng.eval_batch(Xc)
            rate1, _, n1, dt1, _, _, _ = cpu_port_rate(synth, wl, bits, d, r_max, min(3.0, args.cpu_seconds / 4), threads=1)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": nthr, "kind": "port",
                                    "sample": f"{n} candidates of the same workload in {dt:.1f} s",
                                    "value_1_thread": rate1, "sample_1_thread": f"{n1} candidates in {dt1:.1f} s",
                                    "parity_on_sample": bool(np.array_equal(got["count"], ref["count"]) and
                                                             np.array_equal(got["obj"], ref["obj"]))}
        print(json.dumps(line))
    eng.close()
    if c.world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
