"""CoverageEngine -- a thin object wrapper over one libcoverage_cuda handle (one GPU, one stream).

All coverage arithmetic happens in the CUDA kernels behind the C ABI (include/coverage_cuda.h);
this class only marshals NumPy buffers.  Citations are relative to /root/reference/.
"""
from __future__ import annotations

import ctypes as C
import functools
import math

import numpy as np

from . import _lib
from ._lib import CoverageError, lib

TAN_HALF_FOV_DEFAULT = math.tan((100 / 180 * math.pi) / 2)  # FOV = 100/180*pi, src/FullSimulation.jl:735


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _list_order(fn):
    """A horizon method with the keyword list_order: True runs the call with COV_OPT_LIST_ORDER_HORIZON at 1, so that
    it accepts a store whose area depends on the list order (cov_grid_info.area_exact == 0), and puts the handle's
    previous value back afterwards, also when the call raises; False leaves the option as it is."""
    @functools.wraps(fn)
    def call(self, *args, list_order: bool = False, **kwargs):
        if not list_order:
            return fn(self, *args, **kwargs)
        prev = self.get_option(_lib.OPT_LIST_ORDER_HORIZON)
        self.set_option(_lib.OPT_LIST_ORDER_HORIZON, 1)
        try:
            return fn(self, *args, **kwargs)
        finally:
            self.set_option(_lib.OPT_LIST_ORDER_HORIZON, prev)
    return call


class PinnedArray:
    """A NumPy view over pinned host memory obtained from cov_host_alloc (freed with the engine
    or explicitly).  cov_eval_batch DMA-copies pinned buffers in place, without staging."""

    def __init__(self, engine: "CoverageEngine", shape, dtype):
        self._engine = engine
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        engine._check(lib.cov_host_alloc(engine._h, max(n, 1), C.byref(p)))
        self._p = p
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._p is not None and self._engine._h is not None:
            self.array = None
            lib.cov_host_free(self._engine._h, self._p)
        self._p = None


class CoverageEngine:
    """One device-resident cell store + closure parameters + evaluation entry points."""

    def __init__(self, device: int = 0):
        self._h = None
        h = C.c_void_p()
        rc = lib.cov_create(int(device), C.byref(h))
        if rc != _lib.COV_OK:
            raise CoverageError(rc, lib.cov_last_error(None).decode())
        self._h = h
        self.device = int(device)
        self.N = None
        self._pinned = []
        # Who configured the closure parameters last: every set_params() clears it, and a caller that wants
        # to skip redundant uploads stores its own token here afterwards and compares before each use
        # (several objectives / constraints share one engine and must not run on each other's r_max).
        self.param_owner = None

    # ---- plumbing ----
    def _check(self, rc: int):
        if rc != _lib.COV_OK:
            raise CoverageError(rc, lib.cov_last_error(self._h).decode())

    def close(self):
        if self._h is not None:
            for p in self._pinned:
                p.free()
            self._pinned = []
            lib.cov_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def handle(self):
        return self._h

    def set_option(self, option: int, value: int):
        self._check(lib.cov_set_option(self._h, option, int(value)))

    def get_option(self, option: int) -> int:
        v = C.c_int64()
        self._check(lib.cov_get_option(self._h, option, C.byref(v)))
        return v.value

    def pinned(self, shape, dtype=np.float64) -> np.ndarray:
        p = PinnedArray(self, shape, dtype)
        self._pinned.append(p)
        return p.array

    # ---- cell store ----
    def set_grid_bits(self, bits: np.ndarray, nx: int, ny: int, dx: float, dy: float, weight=None):
        """bits: (ny, ceil(nx/32)) uint32; bit b of word w of row j-1 is cell i = 32w+b+1."""
        bits = np.ascontiguousarray(bits, dtype=np.uint32)
        if bits.size != ny * ((nx + 31) // 32):
            raise ValueError("bits must hold ny * ceil(nx/32) words")
        w = dx * dy if weight is None else weight
        self._check(lib.cov_set_grid_bits(self._h, nx, ny, dx, dy, _ptr(bits), w))

    def set_grid_cells(self, mult: np.ndarray, nx: int, ny: int, dx: float, dy: float, cls=None,
                       class_weight=None):
        """mult/cls: nx*ny bytes indexed (i-1) + nx*(j-1)."""
        mult = np.ascontiguousarray(mult, dtype=np.uint8).ravel()
        if mult.size != nx * ny:
            raise ValueError("mult must hold nx*ny bytes")
        if cls is not None:
            cls = np.ascontiguousarray(cls, dtype=np.uint8).ravel()
            if cls.size != nx * ny:
                raise ValueError("cls must hold nx*ny bytes")
        cw = _f64([dx * dy] if class_weight is None else class_weight)
        self._check(lib.cov_set_grid_cells(self._h, nx, ny, dx, dy, _ptr(mult), _ptr(cls), cw.size, _ptr(cw)))

    def set_grid_full(self, nx: int, ny: int, dx: float, dy: float):
        """createPOI(dx, dy, nx, ny) on the device (src/AreaCoverageCalculation.jl:11-21)."""
        self._check(lib.cov_set_grid_full(self._h, nx, ny, dx, dy))

    def set_points(self, pts5: np.ndarray, nx: int, ny: int, dx: float, dy: float):
        """The reference's own list layout: P x 5 [x, y, area, weight, covered]."""
        pts5 = _f64(pts5).reshape(-1, 5)
        self._check(lib.cov_set_points(self._h, _ptr(pts5), pts5.shape[0], nx, ny, dx, dy))

    def add_points(self, pts5: np.ndarray):
        pts5 = _f64(pts5).reshape(-1, 5)
        self._check(lib.cov_add_points(self._h, _ptr(pts5), pts5.shape[0]))

    def grid_info(self) -> dict:
        gi = _lib.GridInfo()
        self._check(lib.cov_get_grid_info(self._h, C.byref(gi)))
        return {f: getattr(gi, f) for f, _ in _lib.GridInfo._fields_}

    def class_weights(self) -> list:
        """Weight of every class as the device numbers them (the k of `class_count[:, k]`)."""
        n = self.grid_info()["n_classes"]
        w = (C.c_double * max(n, 1))()
        self._check(lib.cov_get_class_weights(self._h, w, n))
        return [float(w[k]) for k in range(n)]

    def grid_cells(self) -> np.ndarray:
        gi = self.grid_info()
        out = np.empty(gi["nx"] * gi["ny"], dtype=np.uint8)
        self._check(lib.cov_get_grid_cells(self._h, _ptr(out)))
        return out

    def remove_covered(self, xyR) -> int:
        """rmvCoveredPOI (src/CellFunctions.jl:81-108) on the device-resident store."""
        xyR = _f64(xyR).ravel()
        removed = C.c_int64()
        self._check(lib.cov_remove_covered(self._h, _ptr(xyR), xyR.size // 3, C.byref(removed)))
        return removed.value

    def covered_mask(self, x) -> np.ndarray:
        x = _f64(x).ravel()
        gi = self.grid_info()
        out = np.empty(gi["nx"] * gi["ny"], dtype=np.uint8)
        self._check(lib.cov_covered_mask(self._h, _ptr(x), _ptr(out)))
        return out

    # ---- forest-fire automaton (src/DynamicArea.jl) ----
    def fire_init(self, state: np.ndarray, nx: int, ny: int, dx: float, dy: float, push_initial: bool = True):
        """state: nx*ny bytes (0 EMPTY, 1 TREE, 2 FIRE) indexed (i-1) + nx*(j-1)."""
        state = np.ascontiguousarray(state, dtype=np.uint8).ravel()
        if state.size != nx * ny:
            raise ValueError("state must hold nx*ny bytes")
        self._check(lib.cov_fire_init(self._h, nx, ny, dx, dy, _ptr(state), 1 if push_initial else 0))

    def fire_step(self, wind_speed: float, wind_direction: float, prob_spread: float, seed: int, step: int,
                  append: bool = True) -> int:
        n = C.c_int64()
        self._check(lib.cov_fire_step(self._h, wind_speed, wind_direction, prob_spread, seed, step,
                                      1 if append else 0, C.byref(n)))
        return n.value

    def fire_state(self) -> np.ndarray:
        gi = self.grid_info()
        out = np.empty(gi["nx"] * gi["ny"], dtype=np.uint8)
        self._check(lib.cov_fire_get_state(self._h, _ptr(out)))
        return out

    # ---- parameters ----
    def set_params(self, N: int, r_max, penalty_scale: float = 1e5, prev_xyR=None, d_lim=None,
                   tan_half_fov: float = TAN_HALF_FOV_DEFAULT, sep_min: float = 0.0, use_cons7: bool = False):
        r_max = _f64(r_max).ravel()
        if r_max.size != N:
            raise ValueError("r_max must have N entries")
        if prev_xyR is not None:
            prev_xyR = _f64(prev_xyR).ravel()
            if prev_xyR.size != 3 * N:
                raise ValueError("prev_xyR must have 3N entries")
            d_lim = _f64(np.broadcast_to(np.asarray(d_lim, dtype=np.float64), (N,)))
        self._check(lib.cov_set_params(self._h, N, _ptr(r_max), penalty_scale, _ptr(prev_xyR),
                                       _ptr(d_lim) if prev_xyR is not None else None, tan_half_fov,
                                       float(sep_min), 1 if use_cons7 else 0))
        self.N = int(N)
        self.param_owner = None

    # ---- evaluation ----
    def eval_batch(self, X, want_count=True, want_feasible=True, want_class_count=False,
                   want_progressive=False, out=None):
        """X: (B, 3N) float64, rows [x;y;R].  Returns dict(obj, count, feasible, ...)."""
        X = _f64(X)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        if self.N is None or X.shape[1] != 3 * self.N:
            raise ValueError("X must be (B, 3N) with the N given to set_params")
        B = X.shape[0]
        res = out if out is not None else {}
        if "obj" not in res:
            res["obj"] = np.empty(B, dtype=np.float64)
        if want_count and "count" not in res:
            res["count"] = np.empty(B, dtype=np.int64)
        if want_feasible and "feasible" not in res:
            res["feasible"] = np.empty(B, dtype=np.uint8)
        if want_class_count or want_progressive:
            ncls = self.grid_info()["n_classes"]
            if want_class_count and "class_count" not in res:
                res["class_count"] = np.empty((B, ncls), dtype=np.int64)
            if want_progressive and "progressive" not in res:
                res["progressive"] = np.empty(B, dtype=np.float64)
            self._check(lib.cov_eval_batch_ex(self._h, _ptr(X), B, _ptr(res["obj"]), _ptr(res.get("count")),
                                              _ptr(res.get("feasible")), _ptr(res.get("class_count")),
                                              _ptr(res.get("progressive"))))
        else:
            self._check(lib.cov_eval_batch(self._h, _ptr(X), B, _ptr(res["obj"]), _ptr(res.get("count")),
                                           _ptr(res.get("feasible"))))
        return res

    def eval_batch_best(self, X, barrier: bool = True, out=None):
        """cov_eval_batch_best: the per-candidate outputs of eval_batch plus the poll winner
        (best objective, 0-based index; (inf, -1) when the barrier rejects everything), reduced on the device."""
        X = _f64(X)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        if self.N is None or X.shape[1] != 3 * self.N:
            raise ValueError("X must be (B, 3N) with the N given to set_params")
        B = X.shape[0]
        res = out if out is not None else {}
        if "obj" not in res:
            res["obj"] = np.empty(B, dtype=np.float64)
        if "count" not in res:
            res["count"] = np.empty(B, dtype=np.int64)
        if "feasible" not in res:
            res["feasible"] = np.empty(B, dtype=np.uint8)
        bo, bi = C.c_double(), C.c_int64()
        self._check(lib.cov_eval_batch_best(self._h, _ptr(X), B, _ptr(res["obj"]), _ptr(res["count"]),
                                            _ptr(res["feasible"]), 1 if barrier else 0, C.byref(bo), C.byref(bi)))
        res["best"] = (bo.value, bi.value)
        return res

    _PACKS = {np.dtype(np.float32): _lib.PACK_F32, np.dtype(np.int32): _lib.PACK_I32, np.dtype(np.int16): _lib.PACK_I16}

    def eval_batch_packed(self, Q, granularity: float = 1.0, want_count=True, want_feasible=True, best=False,
                          barrier: bool = True, out=None):
        """cov_eval_batch_packed: candidates on a mesh, sent as int16 / int32 mesh indices (value = q * granularity)
        or float32 values -- a quarter or half of the bytes over PCIe, the same doubles in the kernels.
        Q: (B, 3N) of dtype int16, int32 or float32.  best=True adds res["best"] = (objective, index)."""
        Q = np.ascontiguousarray(Q)
        if Q.dtype not in self._PACKS:
            raise TypeError("Q must be int16, int32 or float32")
        if Q.ndim == 1:
            Q = Q.reshape(1, -1)
        if self.N is None or Q.shape[1] != 3 * self.N:
            raise ValueError("Q must be (B, 3N) with the N given to set_params")
        B = Q.shape[0]
        res = out if out is not None else {}
        if "obj" not in res:
            res["obj"] = np.empty(B, dtype=np.float64)
        if want_count and "count" not in res:
            res["count"] = np.empty(B, dtype=np.int64)
        if want_feasible and "feasible" not in res:
            res["feasible"] = np.empty(B, dtype=np.uint8)
        bo, bi = C.c_double(), C.c_int64()
        self._check(lib.cov_eval_batch_packed(self._h, _ptr(Q), self._PACKS[Q.dtype], float(granularity), B,
                                              _ptr(res["obj"]), _ptr(res.get("count")), _ptr(res.get("feasible")),
                                              1 if barrier else 0, C.byref(bo) if best else None,
                                              C.byref(bi) if best else None))
        if best:
            res["best"] = (bo.value, bi.value)
        return res

    def eval_one(self, x) -> float:
        """AreaMaxObjective(x) for one candidate (src/TDM_STATIC_opt.jl:83-98)."""
        x = _f64(x).ravel()
        if self.N is None or x.size != 3 * self.N:
            raise ValueError("x must have 3N entries")
        v = C.c_double()
        self._check(lib.cov_eval_one(self._h, _ptr(x), C.byref(v)))
        return v.value

    def mads_solve(self, x0, n_iter: int = 100, granularity: float = 1.0, seed: int = 0):
        """One MADS solve in native code (cov_mads_solve). Returns (x, objective, stats dict)."""
        x0 = _f64(x0).ravel()
        if self.N is None or x0.size != 3 * self.N:
            raise ValueError("x0 must have 3N entries")
        out = np.empty_like(x0)
        obj = C.c_double()
        st = (C.c_int64 * 4)()
        self._check(lib.cov_mads_solve(self._h, _ptr(x0), int(n_iter), float(granularity), int(seed) & (2**64 - 1),
                                       _ptr(out), C.byref(obj), st))
        return out, obj.value, {"iterations": st[0], "evaluations": st[1], "batches": st[2], "successes": st[3]}

    def mads_solve_batch(self, X0, n_iter: int = 100, granularity: float = 1.0, seed: int = 0):
        """S independent MADS solves in one launch on the device (cov_mads_solve_batch): solve k starts at X0[k] and
        draws its directions from the Philox key seed + k.  Returns (X S x 3N, objectives S, stats) with stats a dict
        of per-solve int64 arrays: iterations, evaluations, successes, converged."""
        return self._mads_batch(lib.cov_mads_solve_batch, X0, n_iter, granularity, seed)

    def mads_solve_batch_region(self, X0, n_iter: int = 100, granularity: float = 1.0, seed: int = 0):
        """mads_solve_batch on the grid-free static objective of eval_region_batch (cov_mads_solve_batch_region)."""
        return self._mads_batch(lib.cov_mads_solve_batch_region, X0, n_iter, granularity, seed)

    def _mads_batch(self, fn, X0, n_iter, granularity, seed):
        X0 = _f64(X0)
        if X0.ndim == 1:
            X0 = X0.reshape(1, -1)
        if self.N is None or X0.ndim != 2 or X0.shape[1] != 3 * self.N:
            raise ValueError("X0 must be (S, 3N) with the N given to set_params")
        S = X0.shape[0]
        X = np.empty_like(X0)
        obj = np.empty(S, dtype=np.float64)
        st = np.empty((S, 4), dtype=np.int64)
        self._check(fn(self._h, _ptr(X0), S, int(n_iter), float(granularity), int(seed) & (2**64 - 1), _ptr(X),
                       _ptr(obj), _ptr(st)))
        names = ("iterations", "evaluations", "successes", "converged")
        return X, obj, {name: st[:, q].copy() for q, name in enumerate(names)}

    @_list_order
    def run_horizon(self, x_start, T: int, S: int = 1, spread: float = 3.0, n_iter: int = 100,
                    granularity: float = 1.0, seed: int = 0, boxes=None, h_focus: float = 15.0,
                    h_max: float = 30.0):
        """T timesteps of FullSimulation's MADS loop on the device in one call (cov_run_horizon): per timestep
        rmvCoveredPOI of the current swarm, the r_max rule near the boxes (K x 4 rows x_LB, x_UB, y_LB, y_UB; None:
        off), cons3 from the current swarm, S solves from the swarm and S - 1 perturbations of it, the best one as
        the next swarm.  Needs set_params with prev_xyR.  Returns (X (T, 3N), obj (T,), stats, step_ms (T,)) with
        stats a dict of int64 arrays: winner, evaluations, feasible, removed.  The r_max and previous swarm of the
        last timestep stay set on the engine.  list_order=True (keyword, on this method and on run_horizon_points and
        the two ensembles) also accepts a store whose area depends on the list order (non-dyadic weights), replaying
        the reference's list-order sum on the device (COV_OPT_LIST_ORDER_HORIZON for this call only)."""
        return self._horizon(lib.cov_run_horizon, x_start, T, 4, S, spread, n_iter, granularity, seed, boxes, h_focus,
                             h_max, ())

    @_list_order
    def run_horizon_points(self, x_start, appends, S: int = 1, spread: float = 3.0, n_iter: int = 100,
                           granularity: float = 1.0, seed: int = 0, boxes=None, h_focus: float = 15.0,
                           h_max: float = 30.0):
        """run_horizon with the reference's fire list (cov_run_horizon_points): appends is a list of T arrays
        (n_t x 5 reference 5-tuples), timestep t appending appends[t-1] before its rmvCoveredPOI (update_POI's push!).
        Returns (X, obj, stats, step_ms, last_removed): stats gains "appended"; last_removed (nx*ny int32, indexed
        (i-1) + nx*(j-1)) holds the last timestep that removed entries from each cell, 0 if none."""
        rows = [_f64(a).reshape(-1, 5) for a in appends]
        offsets = np.zeros(len(rows) + 1, dtype=np.int64)
        offsets[1:] = np.cumsum([r.shape[0] for r in rows], dtype=np.int64)
        pts = np.concatenate(rows) if offsets[-1] else None
        gi = self.grid_info()
        last = np.zeros(gi["nx"] * gi["ny"], dtype=np.int32)
        out = self._horizon(lib.cov_run_horizon_points, x_start, len(rows), 5, S, spread, n_iter, granularity, seed,
                            boxes, h_focus, h_max, (_ptr(pts), _ptr(offsets)), (_ptr(last),))
        return out + (last,)

    def run_horizon_fire(self, x_start, fire_steps, wind_speed: float, wind_direction: float, prob_spread: float,
                         fire_seed: int, first_step: int, S: int = 1, spread: float = 3.0, n_iter: int = 100,
                         granularity: float = 1.0, seed: int = 0, boxes=None, h_focus: float = 15.0,
                         h_max: float = 30.0):
        """run_horizon with the device automaton (cov_run_horizon_fire): timestep t first runs fire_steps[t-1] steps
        of fire_step(append=True), numbered from first_step.  Returns (X, obj, stats, step_ms) with stats["appended"]
        the entries each timestep's steps pushed."""
        fs = np.ascontiguousarray(fire_steps, dtype=np.int64).ravel()
        return self._horizon(lib.cov_run_horizon_fire, x_start, fs.size, 5, S, spread, n_iter, granularity, seed,
                             boxes, h_focus, h_max, (_ptr(fs), float(wind_speed), float(wind_direction),
                                                     float(prob_spread), int(fire_seed) & (2**64 - 1), int(first_step)))

    @_list_order
    def run_horizon_ensemble(self, x_starts, T: int, S: int = 1, spread: float = 3.0, n_iter: int = 100,
                             granularity: float = 1.0, seed: int = 0, boxes=None, h_focus: float = 15.0,
                             h_max: float = 30.0, want_cells: bool = False):
        """E independent run_horizon scenarios in one call (cov_run_horizon_ensemble), each on a private copy of the
        engine's current store and parameters: scenario e starts from x_starts[e] ((E, 3N)) and equals run_horizon
        with seed + e * T * S.  The engine is left unchanged.  Returns (X (E, T, 3N), obj (E, T), stats, step_ms (T,))
        with stats a dict of (E, T) int64 arrays (run_horizon's), and with want_cells=True also cells (E, nx*ny), the
        multiplicities each scenario leaves (grid_cells after the equivalent run_horizon)."""
        X0 = _f64(x_starts)
        if X0.ndim == 1:
            X0 = X0.reshape(1, -1)
        if self.N is None or X0.ndim != 2 or X0.shape[1] != 3 * self.N:
            raise ValueError("x_starts must be (E, 3N) with the N given to set_params")
        E, T, n = X0.shape[0], max(int(T), 0), 3 * self.N
        B = np.zeros((0, 4)) if boxes is None else _f64(boxes).reshape(-1, 4)
        X = np.empty((E, T, n))
        obj = np.empty((E, T))
        st = np.empty((E, T, 4), dtype=np.int64)
        ms = np.empty(T)
        cells = None
        if want_cells:
            gi = self.grid_info()
            cells = np.empty((E, gi["nx"] * gi["ny"]), dtype=np.uint8)
        self._check(lib.cov_run_horizon_ensemble(self._h, _ptr(X0), E, int(T), int(S), float(spread), int(n_iter),
                                                 float(granularity), int(seed) & (2**64 - 1),
                                                 _ptr(B) if len(B) else None, len(B), float(h_focus), float(h_max),
                                                 _ptr(X), _ptr(obj), _ptr(st), _ptr(ms), _ptr(cells)))
        names = ("winner", "evaluations", "feasible", "removed")
        out = (X, obj, {name: st[:, :, q].copy() for q, name in enumerate(names)}, ms)
        return out + (cells,) if want_cells else out

    def run_horizon_fire_ensemble(self, x_starts, fire_steps, winds, fire_seed: int, first_step: int,
                                  fire_seed_stride: int = 1, S: int = 1, spread: float = 3.0, n_iter: int = 100,
                                  granularity: float = 1.0, seed: int = 0, boxes=None, h_focus: float = 15.0,
                                  h_max: float = 30.0, want_cells: bool = False, want_states: bool = False):
        """E independent run_horizon_fire scenarios in one call (cov_run_horizon_fire_ensemble), each on a private copy
        of the engine's current store, parameters and automaton state: scenario e starts from x_starts[e] ((E, 3N)),
        with the wind winds[e] ((E, 3) rows wind_speed, wind_direction, prob_spread, or one (3,) row for every
        scenario), and equals run_horizon_fire with seed + e * T * S and fire_seed + e * fire_seed_stride (stride 1:
        independent fires, 0: the same fire).  The engine is left unchanged.  Returns (X (E, T, 3N), obj (E, T), stats,
        step_ms (T,)) with stats a dict of (E, T) int64 arrays (run_horizon_fire's, "appended" included), then with
        want_cells=True cells (E, nx*ny), the multiplicities each scenario leaves, and with want_states=True states
        (E, nx*ny), the automaton state each scenario leaves (fire_state's layout)."""
        X0 = _f64(x_starts)
        if X0.ndim == 1:
            X0 = X0.reshape(1, -1)
        if self.N is None or X0.ndim != 2 or X0.shape[1] != 3 * self.N:
            raise ValueError("x_starts must be (E, 3N) with the N given to set_params")
        E, n = X0.shape[0], 3 * self.N
        fs = np.ascontiguousarray(fire_steps, dtype=np.int64).ravel()
        W = _f64(winds)
        if W.shape == (3,):
            W = np.repeat(W[None], E, axis=0)
        if W.shape != (E, 3):
            raise ValueError("winds must be (E, 3) or (3,): wind_speed, wind_direction, prob_spread")
        W = np.ascontiguousarray(W)
        T = fs.size
        B = np.zeros((0, 4)) if boxes is None else _f64(boxes).reshape(-1, 4)
        X = np.empty((E, T, n))
        obj = np.empty((E, T))
        st = np.empty((E, T, 5), dtype=np.int64)
        ms = np.empty(T)
        gi = self.grid_info() if want_cells or want_states else None
        cells = np.empty((E, gi["nx"] * gi["ny"]), dtype=np.uint8) if want_cells else None
        states = np.empty((E, gi["nx"] * gi["ny"]), dtype=np.uint8) if want_states else None
        self._check(lib.cov_run_horizon_fire_ensemble(
            self._h, _ptr(X0), E, T, int(S), float(spread), int(n_iter), float(granularity), int(seed) & (2**64 - 1),
            _ptr(B) if len(B) else None, len(B), float(h_focus), float(h_max), _ptr(fs), _ptr(W),
            int(fire_seed) & (2**64 - 1), int(fire_seed_stride) & (2**64 - 1), int(first_step), _ptr(X), _ptr(obj),
            _ptr(st), _ptr(ms), _ptr(cells), _ptr(states)))
        names = ("winner", "evaluations", "feasible", "removed", "appended")
        out = (X, obj, {name: st[:, :, q].copy() for q, name in enumerate(names)}, ms)
        return out + tuple(a for a, want in ((cells, want_cells), (states, want_states)) if want)

    @_list_order
    def run_horizon_points_ensemble(self, x_starts, schedules, list_of=None, S: int = 1, spread: float = 3.0,
                                    n_iter: int = 100, granularity: float = 1.0, seed: int = 0, boxes=None,
                                    h_focus: float = 15.0, h_max: float = 30.0, want_cells: bool = False,
                                    want_last_removed: bool = False):
        """E independent run_horizon_points scenarios in one call (cov_run_horizon_points_ensemble), each on a private
        copy of the engine's current store and parameters: schedules holds L fire schedules (forecasts), each a list of
        T arrays (n_t x 5 reference 5-tuples) as run_horizon_points takes them, all with the same T; scenario e starts
        from x_starts[e] ((E, 3N)), appends schedule list_of[e] (default: schedule 0 for every scenario) and equals
        run_horizon_points with seed + e * T * S.  The engine is left unchanged.  Returns (X (E, T, 3N), obj (E, T),
        stats, step_ms (T,)) with stats a dict of (E, T) int64 arrays (run_horizon_points'), then with want_cells=True
        cells (E, nx*ny), the multiplicities each scenario leaves, and with want_last_removed=True last_removed
        (E, nx*ny int32), row e what run_horizon_points returns as last_removed for scenario e."""
        X0 = _f64(x_starts)
        if X0.ndim == 1:
            X0 = X0.reshape(1, -1)
        if self.N is None or X0.ndim != 2 or X0.shape[1] != 3 * self.N:
            raise ValueError("x_starts must be (E, 3N) with the N given to set_params")
        E, n = X0.shape[0], 3 * self.N
        if len(schedules) < 1:
            raise ValueError("schedules must hold at least one schedule")
        T = len(schedules[0])
        if any(len(s) != T for s in schedules):
            raise ValueError("every schedule must have the same number of timesteps")
        rows = [_f64(a).reshape(-1, 5) for s in schedules for a in s]  # schedule-major: schedule l, timestep t
        L = len(schedules)
        offsets = np.zeros(L * T + 1, dtype=np.int64)
        offsets[1:] = np.cumsum([r.shape[0] for r in rows], dtype=np.int64)
        pts = np.ascontiguousarray(np.concatenate(rows)) if offsets[-1] else None
        lo = np.zeros(E, dtype=np.int64) if list_of is None else np.ascontiguousarray(list_of, dtype=np.int64)
        if lo.shape != (E,) or (E and (lo.min() < 0 or lo.max() >= L)):
            raise ValueError("list_of must hold E schedule indices in [0, L)")
        B = np.zeros((0, 4)) if boxes is None else _f64(boxes).reshape(-1, 4)
        X = np.empty((E, T, n))
        obj = np.empty((E, T))
        st = np.empty((E, T, 5), dtype=np.int64)
        ms = np.empty(T)
        gi = self.grid_info() if want_cells or want_last_removed else None
        cells = np.empty((E, gi["nx"] * gi["ny"]), dtype=np.uint8) if want_cells else None
        last = np.empty((E, gi["nx"] * gi["ny"]), dtype=np.int32) if want_last_removed else None
        self._check(lib.cov_run_horizon_points_ensemble(
            self._h, _ptr(X0), E, T, int(S), float(spread), int(n_iter), float(granularity), int(seed) & (2**64 - 1),
            _ptr(B) if len(B) else None, len(B), float(h_focus), float(h_max), _ptr(pts), _ptr(offsets), L, _ptr(lo),
            _ptr(X), _ptr(obj), _ptr(st), _ptr(ms), _ptr(cells), _ptr(last)))
        names = ("winner", "evaluations", "feasible", "removed", "appended")
        out = (X, obj, {name: st[:, :, q].copy() for q, name in enumerate(names)}, ms)
        return out + tuple(a for a, want in ((cells, want_cells), (last, want_last_removed)) if want)

    def _horizon(self, fn, x_start, T, cols, S, spread, n_iter, granularity, seed, boxes, h_focus, h_max, source,
                 tail=(), names=("winner", "evaluations", "feasible", "removed", "appended")):
        x_start = _f64(x_start).ravel()
        if self.N is None or x_start.size != 3 * self.N:
            raise ValueError("x_start must have 3N entries")
        B = np.zeros((0, 4)) if boxes is None else _f64(boxes).reshape(-1, 4)
        T = int(T)
        X = np.empty((max(T, 0), 3 * self.N))
        obj = np.empty(max(T, 0))
        st = np.empty((max(T, 0), cols), dtype=np.int64)
        ms = np.empty(max(T, 0))
        self.param_owner = None  # r_max and the previous swarm change on the device
        self._check(fn(self._h, _ptr(x_start), T, int(S), float(spread), int(n_iter), float(granularity),
                       int(seed) & (2**64 - 1), _ptr(B) if len(B) else None, len(B), float(h_focus), float(h_max),
                       *source, _ptr(X), _ptr(obj), _ptr(st), _ptr(ms), *tail))
        return X, obj, {name: st[:, q].copy() for q, name in enumerate(names[:cols])}, ms

    # ---- grid-free static objective ----
    def set_region(self, x_lo: float, y_lo: float, x_hi: float, y_hi: float, covered=None):
        """The domain rectangle and the discs already covered (cov_set_region): covered is M x 3 rows (x, y, R), or
        None for none."""
        C3 = np.zeros((0, 3)) if covered is None else _f64(covered).reshape(-1, 3)
        xyR = np.ascontiguousarray(C3.T).ravel()  # [x_1..x_M, y_1..y_M, R_1..R_M]
        self._check(lib.cov_set_region(self._h, float(x_lo), float(y_lo), float(x_hi), float(y_hi),
                                       _ptr(xyR) if len(C3) else None, len(C3)))

    def run_horizon_region(self, x_start, T: int, S: int = 1, spread: float = 3.0, n_iter: int = 100,
                           granularity: float = 1.0, seed: int = 0, boxes=None, h_focus: float = 15.0,
                           h_max: float = 30.0):
        """run_horizon on the grid-free static objective (cov_run_horizon_region): per timestep the current swarm's
        discs with R > 0 join the region's covered set, then the r_max rule, cons3 from the current swarm and S
        mads_solve_batch_region solves, the best one as the next swarm.  Needs set_region and set_params with
        prev_xyR.  Returns (X (T, 3N), obj (T,), stats, step_ms (T,)) with stats a dict of int64 arrays: winner,
        evaluations, feasible, arcs (of the covered set's boundary at each timestep).  The covered set, its arcs and the
        parameters of the last timestep stay set on the engine; a call that raises leaves the region and the parameters
        as they were."""
        return self._horizon(lib.cov_run_horizon_region, x_start, T, 4, S, spread, n_iter, granularity, seed, boxes,
                             h_focus, h_max, (), names=("winner", "evaluations", "feasible", "arcs"))

    def eval_region_batch(self, X, want_area=True, want_feasible=True, best=False, barrier: bool = True):
        """cov_eval_region_batch: dict(obj, area, feasible) for every row of X (B, 3N), with best=True also
        res["best"] = (objective, index) of the poll winner."""
        X = _f64(X)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        if self.N is None or X.shape[1] != 3 * self.N:
            raise ValueError("X must be (B, 3N) with the N given to set_params")
        B = X.shape[0]
        res = {"obj": np.empty(B, dtype=np.float64)}
        if want_area:
            res["area"] = np.empty(B, dtype=np.float64)
        if want_feasible:
            res["feasible"] = np.empty(B, dtype=np.uint8)
        bo, bi = C.c_double(), C.c_int64()
        self._check(lib.cov_eval_region_batch(self._h, _ptr(X), B, _ptr(res["obj"]), _ptr(res.get("area")),
                                              _ptr(res.get("feasible")), 1 if barrier else 0,
                                              C.byref(bo) if best else None, C.byref(bi) if best else None))
        if best:
            res["best"] = (bo.value, bi.value)
        return res

    def argmin(self, X, barrier: bool = True):
        X = _f64(X)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        bo, bi = C.c_double(), C.c_int64()
        self._check(lib.cov_argmin(self._h, _ptr(X), X.shape[0], 1 if barrier else 0, C.byref(bo), C.byref(bi)))
        return bo.value, bi.value

    def union_area(self, X, N: int) -> np.ndarray:
        """Exact area of the union of the N discs of every row of X (B, 3N) -- the continuous variant."""
        X = _f64(X).reshape(-1, 3 * N)
        out = np.empty(X.shape[0], dtype=np.float64)
        self._check(lib.cov_union_area_batch(self._h, _ptr(X), X.shape[0], N, _ptr(out)))
        return out

    def eval_batch_device(self, dX: int, B: int, d_obj: int, d_count: int = 0, d_feasible: int = 0):
        """Device pointers (ints); asynchronous on the engine's stream."""
        self._check(lib.cov_eval_batch_device(self._h, C.c_void_p(dX), B, C.c_void_p(d_obj),
                                              C.c_void_p(d_count) if d_count else None,
                                              C.c_void_p(d_feasible) if d_feasible else None))

    def generate_candidates(self, dX: int, B: int, N: int, seed: int, first_index: int = 0, lx=500.0, ly=500.0,
                            h_min=5.0, h_max=30.0, tan_half_fov=TAN_HALF_FOV_DEFAULT):
        self._check(lib.cov_generate_candidates(self._h, C.c_void_p(dX), B, N, seed, first_index, lx, ly, h_min,
                                                h_max, tan_half_fov))

    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._check(lib.cov_device_alloc(self._h, nbytes, C.byref(p)))
        return p.value

    def device_free(self, p: int):
        self._check(lib.cov_device_free(self._h, C.c_void_p(p)))

    def memcpy_h2d(self, dst: int, src: np.ndarray):
        self._check(lib.cov_memcpy_h2d(self._h, C.c_void_p(dst), _ptr(src), src.nbytes))

    def memcpy_d2h(self, dst: np.ndarray, src: int):
        self._check(lib.cov_memcpy_d2h(self._h, _ptr(dst), C.c_void_p(src), dst.nbytes))

    def sync(self):
        self._check(lib.cov_sync(self._h))

    def stream(self) -> int:
        return lib.cov_stream(self._h) or 0

    def set_stream(self, stream: int):
        self._check(lib.cov_set_stream(self._h, C.c_void_p(stream) if stream else None))

    def launch_count(self) -> int:
        return lib.cov_launch_count(self._h)

    def last_kernel_ms(self) -> float:
        v = C.c_double()
        self._check(lib.cov_last_kernel_ms(self._h, C.byref(v)))
        return v.value

    def last_launch(self) -> dict:
        """Shape of the last coverage-kernel launch: kernel (KERNEL_SPAN = small-swarm kernel,
        KERNEL_SPAN_GENERAL = CTA per candidate, ...), grid, block, smem_bytes, band_rows, planes_in_smem."""
        li = _lib.LaunchInfo()
        self._check(lib.cov_last_launch(self._h, C.byref(li)))
        return {f: getattr(li, f) for f, _ in _lib.LaunchInfo._fields_}

    def trace(self) -> np.ndarray:
        """Timeline of the last host-path call under OPT_TRACE: (slices, 4) ms [h2d done, k start, k end, d2h done]."""
        n = lib.cov_get_trace(self._h, None, 0)
        out = np.zeros(n)
        lib.cov_get_trace(self._h, out.ctypes.data_as(C.POINTER(C.c_double)), n)
        return out.reshape(-1, 4)

    def kernel_time_total(self):
        """(summed coverage-kernel device time in ms, launches) since the engine was created."""
        ms, n = C.c_double(), C.c_int64()
        self._check(lib.cov_kernel_time_total(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value


def pack_candidates(X, granularity: float = 1.0, dtype=np.int16) -> np.ndarray:
    """Mesh indices of a Float64 candidate matrix for `eval_batch_packed`, LOSSLESS or not at all: returns
    Q = rint(X / granularity) as `dtype` (int16 / int32) after checking that Q * granularity reproduces every entry
    of X exactly (dtype float32: that (double)(float)x == x); raises ValueError otherwise, naming the first
    offending entry.  Pure NumPy (no device): the check costs more than the PCIe bytes it saves, so a caller that
    works in mesh indices anyway (a MADS poll driver does) should keep them rather than call this per batch."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    dtype = np.dtype(dtype)
    if dtype == np.float32:
        Q = X.astype(np.float32)
        back = Q.astype(np.float64)
    elif dtype in (np.dtype(np.int16), np.dtype(np.int32)):
        if not (granularity > 0 and math.isfinite(granularity)):
            raise ValueError("granularity must be a positive finite number")
        q = np.rint(X / granularity)
        info = np.iinfo(dtype)
        bad = ~((q >= info.min) & (q <= info.max))  # (also catches NaN)
        if bad.any():
            k = np.argwhere(bad)[0]
            raise ValueError(f"entry {tuple(int(v) for v in k)} = {X[tuple(k)]!r} does not fit {dtype.name} mesh indices")
        Q = q.astype(dtype)
        back = Q.astype(np.float64) * granularity
    else:
        raise TypeError("dtype must be int16, int32 or float32")
    same = (back == X) | (np.isnan(back) & np.isnan(X))  # by value: -0.0 packs as +0, which no term of the objective can tell apart
    if not same.all():
        k = np.argwhere(~same)[0]
        raise ValueError(f"entry {tuple(int(v) for v in k)} = {X[tuple(k)]!r} is not on the mesh of granularity "
                         f"{granularity!r} ({dtype.name}): packing would change it")
    return Q


def threshold(R: float) -> float:
    """T(R): sqrt(s) < R  <=>  s < T(R) (the closed form the kernels use)."""
    return lib.cov_threshold(float(R))


def limits() -> dict:
    lim = _lib.Limits()
    lib.cov_get_limits(C.byref(lim))
    return {f: getattr(lim, f) for f, _ in _lib.Limits._fields_}


def device_count() -> int:
    return lib.cov_device_count()
