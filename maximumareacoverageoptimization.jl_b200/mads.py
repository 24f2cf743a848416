"""Batched MADS poll driver -- the caller side of the coverage objective (SURVEY.md 8f-1).

The reference's `TDM_STATIC_opt.optimize` (/root/reference/src/TDM_STATIC_opt.jl:118-222) hands the
objective to DirectSearch.jl, which evaluates ONE trial point per call.  DirectSearch.jl is a
third-party package that is neither vendored nor pinned by the reference (absent from
Project.toml, Manifest.toml git-ignored), and LTMADS draws unseeded random directions, so the MADS
iterates themselves are not reproducible by anyone -- MADS trajectory parity is UNPINNED; only the
settings below and the objective values are.

This driver keeps the reference's call shape and settings

    optimize(input, obj, cons_ext, cons_prog, N_iter) -> (result, runtime)
    * n = len(input) variables, initial point `input`               (:123-124)
    * iteration limit N_iter                                         (:126)
    * granularity 1.0 on every variable                              (:131-137)
    * extreme (barrier) constraints `cons_ext`                       (:151-153)
    * result = feasible incumbent if there is one, else the start    (:165-169)
    * runtime = total wall time of the solve in seconds              (:219)

and restates the published algorithm it needs -- the granular-variable mesh of Audet, Le Digabel &
Tribes, "The mesh adaptive direct search algorithm for granular and discrete variables" (SIAM J.
Optim. 29(2), 2019): poll size Delta_i = a * 10^b with a in {1, 2, 5}, mesh size
delta_i = max(10^(b - |b - b0|), granularity), 2n poll directions from a random Householder matrix
rounded onto the mesh -- but evaluates each poll set as ONE batch through `obj.batch`, with the
extreme constraints fused into the same kernel launch when they carry a `.fuse` description
(create_cons3 / create_cons7 / create_cons8).  Polling is complete (no opportunistic stop): the
whole set is already evaluated when the winner is picked.
"""
from __future__ import annotations

import math
import time

import numpy as np


class _Mesh:
    """Per-variable poll size a*10^b and mesh size (Audet, Le Digabel & Tribes 2019, section 3)."""

    def __init__(self, x0, granularity):
        n = len(x0)
        self.g = np.asarray(granularity, dtype=np.float64) * np.ones(n)
        self.a = np.ones(n)
        self.b = np.zeros(n, dtype=np.int64)
        for i in range(n):
            # initial poll size: about a tenth of |x0_i| (at least 1), on the {1, 2, 5} x 10^b ladder
            target = max(abs(float(x0[i])) / 10.0, 1.0, self.g[i])
            b = int(math.floor(math.log10(target)))
            m = target / 10.0 ** b
            self.a[i] = 1.0 if m < 2 else (2.0 if m < 5 else 5.0)
            self.b[i] = b
        self.b0 = self.b.copy()

    def poll_size(self):
        return np.maximum(self.a * 10.0 ** self.b, self.g)

    def mesh_size(self):
        return np.maximum(10.0 ** (self.b - np.abs(self.b - self.b0)), self.g)

    def enlarge(self):
        for i in range(len(self.a)):
            if self.a[i] == 1.0:
                self.a[i] = 2.0
            elif self.a[i] == 2.0:
                self.a[i] = 5.0
            else:
                self.a[i] = 1.0
                self.b[i] += 1

    def refine(self):
        """Returns False when no variable can be refined any further (every poll size sits at its
        granularity): the mesh has bottomed out."""
        moved = False
        for i in range(len(self.a)):
            if self.g[i] > 0 and self.a[i] * 10.0 ** self.b[i] <= self.g[i]:
                continue
            if self.a[i] == 1.0:
                self.a[i] = 5.0
                self.b[i] -= 1
            elif self.a[i] == 2.0:
                self.a[i] = 1.0
            else:
                self.a[i] = 2.0
            moved = True
        return moved


def _poll_directions(n: int, rho: np.ndarray, rng: np.random.Generator) -> np.ndarray:
    """2n integer mesh directions: columns of a random Householder matrix, each scaled so that its
    largest component spans the poll-to-mesh ratio rho_i, rounded to integers, plus their negatives."""
    v = rng.normal(size=n)
    v /= np.linalg.norm(v)
    H = np.eye(n) - 2.0 * np.outer(v, v)
    D = np.empty((n, n))
    for j in range(n):
        h = H[:, j]
        D[:, j] = np.rint(rho * h / np.max(np.abs(h)))
    D = D[:, np.any(D != 0, axis=0)]
    return np.concatenate([D, -D], axis=1).T  # (<= 2n, n)


def _snap(x, g):
    """Round onto the granular mesh (absolute multiples of the granularity)."""
    return np.where(g > 0, np.rint(x / np.where(g > 0, g, 1.0)) * g, x)


class _Solve:
    """One MADS solve as a state machine: `poll()` hands out the next poll set, `update(P, f)` takes its objective
    values (extreme barrier already applied: +inf where a constraint fails).  `optimize` drives one of these,
    `optimize_multistart` many in lockstep."""

    def __init__(self, x0, g, rng, snap_initial=False):
        self.x0, self.g, self.rng = x0, g, rng
        self.x = _snap(x0, g) if snap_initial else x0.copy()
        self.fx = math.inf
        self.mesh = None
        self.feasible_found = False
        self.done = False
        self.iterations = 0
        self.successes = 0

    def start(self, fx: float):
        self.fx = fx
        self.mesh = _Mesh(self.x, self.g)
        self.feasible_found = math.isfinite(fx)

    def poll(self) -> np.ndarray:
        self.iterations += 1
        n = self.x.size
        delta, Delta = self.mesh.mesh_size(), self.mesh.poll_size()
        D = _poll_directions(n, np.maximum(np.rint(Delta / delta), 1.0), self.rng)
        P = _snap(self.x[None, :] + D * delta[None, :], self.g)
        P = P[np.any(P != self.x[None, :], axis=1)]
        return np.unique(P, axis=0) if len(P) else P

    def update(self, P: np.ndarray, f: np.ndarray):
        k = int(np.argmin(f)) if len(P) else -1
        best = float(f[k]) if len(P) else math.inf
        if best < self.fx or (not self.feasible_found and math.isfinite(best)):
            self.x, self.fx = P[k].copy(), best
            self.feasible_found = True
            self.successes += 1
            self.mesh.enlarge()
        elif not self.mesh.refine():
            self.done = True  # every poll size is down at its granularity: the granular mesh cannot refine

    def result(self) -> np.ndarray:
        return self.x if self.feasible_found else self.x0  # p.x if there is a feasible incumbent, else the start (p.i)


def _flatten_constraints(cons_ext):
    flat = []
    for c in (cons_ext if isinstance(cons_ext, (list, tuple)) else [cons_ext]):
        flat.extend(c if isinstance(c, (list, tuple)) else [c])
    return flat


def _barrier_evaluator(obj, host_cons, stats, cache):
    """P -> objective of every row with the extreme barrier (+inf where a constraint fails), ONE obj.batch call for
    the rows not seen before."""
    def evaluate(P):
        P = np.ascontiguousarray(P, dtype=np.float64)
        keys = [p.tobytes() for p in P]
        f = np.empty(len(P))
        todo = [k for k in range(len(P)) if keys[k] not in cache]
        stats["cache_hits"] += len(P) - len(todo)
        if todo:
            Q = P[todo]
            ok = np.ones(len(Q), dtype=bool)
            for c in host_cons:  # extreme barrier: constraints first, objective only where they hold
                ok &= np.asarray(c.batch(Q), dtype=bool) if hasattr(c, "batch") else np.array([bool(c(q)) for q in Q])
            if hasattr(obj, "batch"):
                try:
                    vals, feas = obj.batch(Q, want_feasible=True)
                    ok &= np.asarray(feas, dtype=bool)
                except TypeError:
                    vals = obj.batch(Q)
                vals = np.asarray(vals, dtype=np.float64)
            else:
                vals = np.array([obj(q) if ok[k] else math.inf for k, q in enumerate(Q)])
            vals = np.where(ok, vals, math.inf)
            stats["evaluations"] += len(Q)
            stats["batches"] += 1
            for k, idx in enumerate(todo):
                cache[keys[idx]] = float(vals[k])
        for k in range(len(P)):
            f[k] = cache[keys[k]]
        return f
    return evaluate


def optimize(input, obj, cons_ext, cons_prog, N_iter, granularity=1.0, seed=None, snap_initial=False,
             return_stats=False, native=None):
    """src/TDM_STATIC_opt.jl:118-222.  `obj`: callable x -> float, preferably with `.batch(X)` (and
    `.fuse(constraints)`, see TDM_STATIC_opt.AreaMaxObjective).  `cons_ext`: extreme constraints
    x -> bool (flat list; nested lists as in FullSimulation.jl:86 `[cons_ext, cons3]` are flattened).
    `cons_prog` is accepted and ignored exactly like the reference does (:154-159 is commented out).
    Returns (result, runtime) -- with return_stats=True also a dict of counters.

    native: True runs the whole solve inside the library (cov_mads_solve: same algorithm and settings, its own
    random stream, no Python between polls); it needs an objective made by createObjective on a list with
    exactly summable weights and constraints that all fuse.  None (default) picks it when that holds."""
    t_start = time.perf_counter()
    if native is not False and hasattr(obj, "native_solver") and np.isscalar(granularity) and not snap_initial:
        solver = obj.native_solver(_flatten_constraints(cons_ext))
        if solver is not None:
            x, fx, st = solver(np.ascontiguousarray(input, dtype=np.float64).ravel(), int(N_iter), float(granularity),
                               0 if seed is None else int(seed))
            runtime = time.perf_counter() - t_start
            st["objective"] = fx
            return (x, runtime, st) if return_stats else (x, runtime)
        if native is True:
            raise ValueError("native MADS needs fusable constraints and exactly summable weights")
    x0 = np.ascontiguousarray(input, dtype=np.float64).ravel().copy()
    n = x0.size
    rng = np.random.default_rng(seed)

    flat = _flatten_constraints(cons_ext)
    host_cons = obj.fuse(flat) if hasattr(obj, "fuse") else flat

    stats = {"iterations": 0, "evaluations": 0, "batches": 0, "cache_hits": 0, "successes": 0}
    evaluate = _barrier_evaluator(obj, host_cons, stats, {})

    g = np.asarray(granularity, dtype=np.float64) * np.ones(n)
    solve = _Solve(x0, g, rng, snap_initial)
    solve.start(float(evaluate(solve.x[None, :])[0]))
    for _ in range(int(N_iter)):
        P = solve.poll()
        solve.update(P, evaluate(P) if len(P) else np.empty(0))
        if solve.done:
            break
    stats["iterations"], stats["successes"] = solve.iterations, solve.successes
    x, fx, feasible_found = solve.x, solve.fx, solve.feasible_found
    result = x if feasible_found else x0  # p.x if there is a feasible incumbent, else the start (p.i)
    runtime = time.perf_counter() - t_start
    stats["objective"] = fx
    if return_stats:
        return result, runtime, stats
    return result, runtime


def optimize_multistart(inputs, obj, cons_ext, cons_prog, N_iter, granularity=1.0, seed=None, return_stats=False,
                        native=False):
    """S independent MADS solves from the rows of `inputs` (S x n), with the settings of `optimize`, advanced in
    LOCKSTEP: at every iteration the poll sets of all the solves still running are concatenated and evaluated in ONE
    `obj.batch` call (S x 2n trial points per launch instead of 2n -- SURVEY.md 8f-1's multi-start swarms: a 30-point
    poll costs the GPU a launch whether it carries 30 candidates or 3 000).  Solve k draws its directions from
    `default_rng(seed + k)`, so its iterates are exactly those of `optimize(inputs[k], ..., seed=seed + k,
    native=False)`; lockstep changes how the work is batched, not what is computed.
    Returns (results S x n, objectives S, runtime) -- results[k] is solve k's feasible incumbent, else its start;
    objectives[k] is +inf where solve k never found a feasible point.  With return_stats=True also a dict of counters
    (iterations = lockstep iterations, batches = obj.batch calls, per_solve_iterations, best = argmin of objectives).

    native=True runs all S solves on the device in ONE launch (cov_mads_solve_batch: the same algorithm and settings,
    solve k seeded seed + k, directions from the library's own Philox stream instead of NumPy's, so the iterates differ
    from native=False); stats["batches"] is 1.  It needs an objective made by createObjective, constraints that all
    fuse and a scalar granularity, and raises ValueError otherwise."""
    t_start = time.perf_counter()
    X0 = np.ascontiguousarray(inputs, dtype=np.float64)
    if X0.ndim != 2 or not len(X0):
        raise ValueError("inputs must be S x n with S >= 1")
    S, n = X0.shape
    flat = _flatten_constraints(cons_ext)
    if native:
        solver = obj.native_batch_solver(flat) if hasattr(obj, "native_batch_solver") else None
        if solver is None or not np.isscalar(granularity):
            raise ValueError("native multistart needs an objective from createObjective, constraints that all fuse and "
                             "a scalar granularity")
        results, objectives, st = solver(X0, int(N_iter), float(granularity), 0 if seed is None else int(seed))
        runtime = time.perf_counter() - t_start
        if return_stats:
            stats = {"iterations": int(st["iterations"].max()), "evaluations": int(st["evaluations"].sum()),
                     "batches": 1, "cache_hits": 0, "successes": int(st["successes"].sum()),
                     "per_solve_iterations": st["iterations"].tolist(), "best": int(np.argmin(objectives))}
            return results, objectives, runtime, stats
        return results, objectives, runtime
    host_cons = obj.fuse(flat) if hasattr(obj, "fuse") else flat
    stats = {"iterations": 0, "evaluations": 0, "batches": 0, "cache_hits": 0, "successes": 0}
    evaluate = _barrier_evaluator(obj, host_cons, stats, {})
    g = np.asarray(granularity, dtype=np.float64) * np.ones(n)
    solves = [_Solve(X0[k].copy(), g, np.random.default_rng(None if seed is None else seed + k)) for k in range(S)]
    for s, f0 in zip(solves, evaluate(np.stack([s.x for s in solves]))):
        s.start(float(f0))
    for _ in range(int(N_iter)):
        active = [s for s in solves if not s.done]
        if not active:
            break
        stats["iterations"] += 1
        polls = [s.poll() for s in active]
        rows = [len(P) for P in polls]
        f = evaluate(np.concatenate(polls)) if sum(rows) else np.empty(0)
        at = 0
        for s, P, m in zip(active, polls, rows):
            s.update(P, f[at:at + m])
            at += m
    results = np.stack([s.result() for s in solves])
    objectives = np.array([s.fx if s.feasible_found else math.inf for s in solves])
    runtime = time.perf_counter() - t_start
    if return_stats:
        stats["successes"] = sum(s.successes for s in solves)
        stats["per_solve_iterations"] = [s.iterations for s in solves]
        stats["best"] = int(np.argmin(objectives))
        return results, objectives, runtime, stats
    return results, objectives, runtime
