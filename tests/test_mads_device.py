"""The device MADS solver (cov_mads_solve_batch): S solves in one launch.

CPU: what nvcc built for it (cuobjdump).  GPU: every iterate against a NumPy restatement of cov_mads_solve's loop
(cov_api.cu) driven by the library's documented direction stream, the objective of every poll set taken from
cov_eval_batch -- X_out, obj_out and the four stats must agree bit for bit; independence of the solves of one
launch; results against the C oracle; the error classes; the Python entry points."""
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

T = math.tan((100 / 180 * math.pi) / 2)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "maximumareacoverageoptimization.jl_b200", "libcoverage_cuda.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
M32 = 0xFFFFFFFF


# ---------------------------------------------------------------- CPU: the compiled kernel
@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_mads_kernel_fits_its_launch_plan():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    mads = {k: v for k, v in usage.items() if "mads_kernel" in k}
    assert len(mads) == 4, sorted(mads)  # mads_kernel<MULTI, PLANES_SMEM, THREADS, CTAS>
    for k, v in mads.items():
        assert v["LOCAL"] == 0 and v["STACK"] <= 128, (k, v)
        threads, ctas = map(int, re.search(r"ILb[01]ELb[01]ELi(\d+)ELi(\d+)E", k).groups())
        assert v["REG"] * threads * ctas <= 65536, (k, v)


# ---------------------------------------------------------------- the host model
def _p10(b: int) -> float:
    b = max(-400, min(400, int(b)))
    try:
        return 10.0 ** b  # the C library's pow, as std::pow in the library
    except OverflowError:
        return math.inf


def _mx(a, b):
    return np.where(a < b, b, a)  # std::max


def directions(synth, key: int, t: int, n: int) -> np.ndarray:
    """Irwin-Hall(12) normals from Philox4x32-10 keyed by `key` (= seed + k mod 2^64), counter (t lo, t hi, i, g),
    normalised with a sequential sum."""
    i = np.arange(n, dtype=np.uint64)
    z = np.zeros(n, dtype=np.uint64)
    s = np.zeros(n, dtype=np.uint64)
    for g in range(3):
        for w in synth._philox(z + np.uint64(t & M32), z + np.uint64(t >> 32), i, z + np.uint64(g), key & M32,
                               (key >> 32) & M32):
            s += w
    v = s.astype(np.float64) * 2.0 ** -32 - 6.0
    nrm = 0.0
    for vi in v.tolist():
        nrm += vi * vi
    return v / math.sqrt(nrm)


class _Model:
    """One solve of cov_mads_solve's loop (cov_api.cu) with the device stream, no cache, no duplicate removal."""

    def __init__(self, synth, x0, g, key):
        self.synth, self.x0, self.x, self.g, self.key = synth, x0, x0.copy(), g, key
        n = x0.size
        self.a, self.b = np.empty(n), np.empty(n, dtype=np.int64)
        for i in range(n):  # cov_api.cu initial_mesh
            target = max(max(abs(float(x0[i])) / 10.0, 1.0), g)
            lb = math.log10(target)  # +Inf for an infinite start, NaN for a NaN one: b clamped to 400, NaN to 0
            b = 0 if lb != lb else (400 if lb == math.inf else min(math.floor(lb), 400))
            mant = target / _p10(b)
            self.a[i], self.b[i] = (1.0 if mant < 2 else (2.0 if mant < 5 else 5.0)), b
        self.b0 = self.b.copy()
        self.it = self.evaluations = self.successes = self.converged = 0
        self.done = False

    def start(self, f0):
        self.fx, self.found, self.evaluations = f0, math.isfinite(f0), 1

    def poll(self):
        n, g = self.x.size, self.g
        with np.errstate(all="ignore"):
            Delta = _mx(self.a * np.array([_p10(b) for b in self.b]), g)
            delta = _mx(np.array([_p10(b - abs(b - b0)) for b, b0 in zip(self.b, self.b0)]), g)
            rho = _mx(np.rint(Delta / delta), 1.0)
            v = directions(self.synth, self.key, self.it, n)
            self.it += 1
            H = np.eye(n) - np.outer(2.0 * v, v)                 # H[i, j] = delta_ij - (2 v_i) v_j
            A = np.abs(H)
            hmax = np.where(A == A, A, 0.0).max(axis=0)          # std::max never picks a NaN
            D = np.rint((rho[:, None] * H) / hmax[None, :])
            P = np.concatenate([self.x[:, None] + D * delta[:, None], self.x[:, None] + (-1.0 * D) * delta[:, None]], 1)
            if g > 0:
                P = np.rint(P / g) * g
            anyd = np.concatenate([np.any(D != 0, axis=0)] * 2)
            keep = anyd & np.any(P != self.x[:, None], axis=0)
        return P.T[keep].copy()

    def update(self, P, f):
        self.evaluations += len(P)
        best, kb = math.inf, -1
        for k, fk in enumerate(f.tolist()):
            if fk < best:
                best, kb = fk, k
        if kb >= 0 and (best < self.fx or (not self.found and math.isfinite(best))):
            self.x, self.fx, self.found = P[kb].copy(), best, True
            self.successes += 1
            for i in range(self.a.size):
                if self.a[i] == 1.0:
                    self.a[i] = 2.0
                elif self.a[i] == 2.0:
                    self.a[i] = 5.0
                else:
                    self.a[i], self.b[i] = 1.0, self.b[i] + 1
        else:
            moved = False
            for i in range(self.a.size):
                if self.g > 0 and self.a[i] * _p10(self.b[i]) <= self.g:
                    continue
                if self.a[i] == 1.0:
                    self.a[i], self.b[i] = 5.0, self.b[i] - 1
                elif self.a[i] == 2.0:
                    self.a[i] = 1.0
                else:
                    self.a[i] = 2.0
                moved = True
            if not moved:
                self.converged, self.done = 1, True


def model_batch(synth, eng, X0, n_iter, g, seed):
    """The S solves in lockstep; each iteration's kept points of all of them in one cov_eval_batch."""
    def barrier(P):
        if not len(P):
            return np.empty(0)
        r = eng.eval_batch(P, want_count=False, want_feasible=True)
        return np.where((r["feasible"] != 0) & (r["obj"] == r["obj"]), r["obj"], math.inf)

    solves = [_Model(synth, X0[k].copy(), g, (seed + k) % 2 ** 64) for k in range(len(X0))]
    for s, f0 in zip(solves, barrier(X0)):
        s.start(float(f0))
    for _ in range(n_iter):
        act = [s for s in solves if not s.done]
        if not act:
            break
        polls = [s.poll() for s in act]
        f = barrier(np.concatenate(polls)) if sum(len(P) for P in polls) else np.empty(0)
        at = 0
        for s, P in zip(act, polls):
            s.update(P, f[at:at + len(P)])
            at += len(P)
    X = np.stack([s.x if s.found else s.x0 for s in solves])
    obj = np.array([s.fx for s in solves])
    st = {"iterations": np.array([s.it for s in solves]), "evaluations": np.array([s.evaluations for s in solves]),
          "successes": np.array([s.successes for s in solves]), "converged": np.array([s.converged for s in solves])}
    return X, obj, st


def assert_same(got, want):
    X, obj, st = got
    Xm, objm, stm = want
    assert np.array_equal(X.view(np.uint64), Xm.view(np.uint64)), np.flatnonzero(np.any(X != Xm, axis=1))[:10]
    assert np.array_equal(obj.view(np.uint64), objm.view(np.uint64)), (obj, objm)
    for name in ("iterations", "evaluations", "successes", "converged"):
        assert np.array_equal(st[name], stm[name]), (name, st[name], stm[name])


# ---------------------------------------------------------------- GPU scenarios
def _starts(rng, x0, S, N, spread=3.0, far=0):
    X0 = np.repeat(x0[None, :], S, axis=0)
    X0[:, :2 * N] += np.rint(rng.normal(0, spread, (S, 2 * N)))
    X0[:far, :N] += 60.0  # beyond cons3's 10 m: infeasible starts
    return X0


def _config1(cov, engine, N=5, d_lim=10.0):
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    engine.set_grid_full(100, 100, 5.0, 5.0)
    engine.set_params(N, np.full(N, 30 * T))
    engine.remove_covered(x0)  # rmvCoveredPOI with the starting swarm, as FullSimulation does
    engine.set_params(N, np.full(N, 30 * T), prev_xyR=x0, d_lim=d_lim, tan_half_fov=T)
    return x0


SCENARIOS = ["c1_cons3", "fire_cons8", "ordered", "gran_half", "gran_zero", "force_exact", "n1", "n64"]


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", SCENARIOS)
def test_bit_for_bit_against_host_model(cov, engine, fire_rows, scenario):
    rng = np.random.default_rng(SCENARIOS.index(scenario) + 1)
    g, n_iter, seed = 1.0, 100, 17
    if scenario in ("c1_cons3", "gran_half", "gran_zero", "force_exact"):
        N = 5
        x0 = _config1(cov, engine, N)
        S = 32 if scenario == "c1_cons3" else 8
        X0 = _starts(rng, x0, S, N, far=4 if scenario == "c1_cons3" else 0)
        if scenario == "gran_half":
            g = 0.5
        elif scenario == "gran_zero":
            g, n_iter = 0.0, 60
            X0 = X0 + rng.random(X0.shape) * 0.01  # off every mesh
        elif scenario == "force_exact":
            engine.set_option(cov.OPT_FORCE_EXACT, 1)
    elif scenario == "fire_cons8":
        N = 5
        engine.set_points(np.concatenate(fire_rows), 100, 100, 5.0, 5.0)
        assert engine.grid_info()["n_planes"] == 2
        engine.set_params(N, np.full(N, 30 * T), sep_min=15.0)
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 330.0)
        X0 = _starts(rng, x0, 16, N, spread=10.0)
        X0[:3, :N], X0[:3, N:2 * N] = 250.0 + np.arange(N) * 5.0, 300.0  # 5 m apart: these starts break cons8
    elif scenario == "ordered":
        N = 5
        pts = np.concatenate(fire_rows[:30]).copy()
        hi = (pts[:, 0] > 240) & (pts[:, 0] < 300)
        pts[hi, 2] = pts[hi, 3] = (30 * T) ** 2 * math.pi  # the high-interest weight: not dyadic
        engine.set_points(pts, 100, 100, 5.0, 5.0)
        assert engine.grid_info()["area_exact"] == 0 and engine.grid_info()["n_classes"] == 2
        engine.set_params(N, np.full(N, 30 * T))
        x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 330.0)
        X0 = _starts(rng, x0, 8, N, spread=8.0)
        n_iter = 60
    elif scenario == "n1":
        N = 1
        x0 = _config1(cov, engine, N)
        X0 = _starts(rng, x0, 8, N)
    else:  # n64: the largest swarm of the launch plan, on a small grid
        N = 64
        engine.set_grid_full(40, 40, 5.0, 5.0)
        engine.set_params(N, np.full(N, 6.0))
        X0 = np.concatenate([np.rint(rng.random((3, 2 * N)) * 200), np.rint(2 + rng.random((3, N)) * 6)], axis=1)
        n_iter = 12
    got = engine.mads_solve_batch(X0, n_iter, g, seed)
    want = model_batch(cov.synth, engine, X0, n_iter, g, seed)
    assert_same(got, want)
    assert got[2]["iterations"].max() >= 1 and got[2]["successes"].sum() > 0
    if scenario == "c1_cons3":
        assert np.any(~np.isfinite(model_batch(cov.synth, engine, X0, 0, g, seed)[1]))  # some starts infeasible
        assert got[2]["converged"].sum() > 0  # some solves bottom out on the integer mesh within 100 iterations


@pytest.mark.gpu
def test_solves_are_independent(cov, engine):
    """Solve k of a launch is the S = 1 call on X0[k] with seed + k, also when there are more solves than resident
    CTAs (persistent CTAs take the later ones from the dispenser)."""
    N = 5
    x0 = _config1(cov, engine, N)
    rng = np.random.default_rng(3)
    S, seed = 2000, 2**64 - 1000  # the keys seed + k wrap around 2^64
    X0 = _starts(rng, x0, S, N, far=50)
    X, obj, st = engine.mads_solve_batch(X0, 100, 1.0, seed)
    for k in (0, 1, 499, 999, 1000, 1337, 1999):
        Xk, objk, stk = engine.mads_solve_batch(X0[k:k + 1], 100, 1.0, (seed + k) % 2**64)
        assert np.array_equal(Xk[0].view(np.uint64), X[k].view(np.uint64)) and objk[0] == obj[k]
        assert all(stk[name][0] == st[name][k] for name in st)
    assert engine.launch_count() >= 8


@pytest.mark.gpu
def test_results_against_the_oracle(cov, orc, engine):
    N = 5
    x0 = _config1(cov, engine, N)
    pts = orc.rmvCoveredPOI(x0, orc.createPOI(5.0, 5.0, 100.0, 100.0))  # the list the engine's store holds
    r_max = np.full(N, 30 * T)
    rng = np.random.default_rng(5)
    X0 = _starts(rng, x0, 64, N, far=6)
    f0 = model_batch(cov.synth, engine, X0, 0, 1.0, 0)[1]
    X, obj, st = engine.mads_solve_batch(X0, 100, 1.0, 0)
    for k in range(len(X0)):
        if math.isfinite(obj[k]):
            assert orc.objective(X[k], r_max, pts)[0] == obj[k]
            assert orc.cons3(X[k], x0, T, np.full(N, 10.0))
            assert np.all(X[k] == np.rint(X[k]))  # on the mesh of granularity 1
            assert obj[k] <= f0[k]
        else:
            assert np.array_equal(X[k], X0[k])
    assert np.isfinite(obj).sum() >= 58
    # n_iter = 0: the starts and their values
    X, obj, st = engine.mads_solve_batch(X0, 0, 1.0, 0)
    assert np.array_equal(X, X0) and np.array_equal(obj, f0)
    assert np.all(st["iterations"] == 0) and np.all(st["evaluations"] == 1) and np.all(st["converged"] == 0)


@pytest.mark.gpu
def test_errors_leave_the_handle_usable(cov, engine):
    L = cov._lib
    lib, h = L.lib, engine.handle
    X0 = np.zeros((2, 15))
    out = np.empty_like(X0)

    def call(X, S, n_iter=10, g=1.0, Xo=out):
        return lib.cov_mads_solve_batch(h, None if X is None else X.ctypes.data, S, n_iter, g, 0,
                                        None if Xo is None else Xo.ctypes.data, None, None)

    assert call(X0, 2) == L.COV_ERR_STATE  # no grid
    engine.set_grid_full(100, 100, 5.0, 5.0)
    assert call(X0, 2) == L.COV_ERR_STATE  # no params
    engine.set_params(5, np.full(5, 30 * T))
    assert call(None, 2) == L.COV_ERR_INVALID
    assert call(X0, 2, Xo=None) == L.COV_ERR_INVALID
    assert call(X0, -1) == L.COV_ERR_INVALID
    assert call(X0, 2, n_iter=-1) == L.COV_ERR_INVALID
    assert call(X0, 2, g=-1.0) == L.COV_ERR_INVALID
    assert call(X0, 2, g=math.nan) == L.COV_ERR_INVALID
    assert call(X0, 0) == L.COV_OK  # nothing to do
    engine.set_params(65, np.full(65, 30 * T))
    with pytest.raises(cov.CoverageError) as e:
        engine.mads_solve_batch(np.zeros((1, 195)), 5)
    assert e.value.code == L.COV_ERR_LIMIT and "64" in e.value.message
    engine.set_grid_full(8192, 8192, 500 / 8192, 500 / 8192)  # one warp's framebuffer: 8 MiB
    engine.set_params(5, np.full(5, 30 * T))
    with pytest.raises(cov.CoverageError) as e:
        engine.mads_solve_batch(np.full((1, 15), 100.0), 5)
    assert e.value.code == L.COV_ERR_LIMIT and "shared memory" in e.value.message
    engine.set_grid_full(100, 100, 5.0, 5.0)
    X = cov.synth.random_candidates(100, 5, seed=1)
    assert np.isfinite(engine.eval_batch(X)["obj"]).all()
    assert engine.mads_solve_batch(X[:3], 5)[1].shape == (3,)


@pytest.mark.gpu
def test_optimize_multistart_native(cov):
    CF, OPT, TC, ACC = cov.CellFunctions, cov.TDM_STATIC_opt, cov.TDM_Constraints, cov.AreaCoverageCalculation
    cells = CF.initialise_POI(CF.Cells(), "static")
    N, FOV = 5, 100 / 180 * math.pi
    r_max = np.full(N, 30.0 * T)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    cells = CF.rmvCoveredPOI(cells, x0)
    obj = OPT.createObjective(cells, N, r_max)
    cons3 = TC.create_cons3(ACC.make_circles(x0), FOV, 10 * np.ones(N))
    X0 = _starts(np.random.default_rng(9), x0, 12, N)
    res, objs, runtime, st = OPT.optimize_multistart(X0, obj, [TC.cons1, cons3], [], 100, seed=40, return_stats=True,
                                                     native=True)
    eng = obj._engine()[1]
    X, o, s = eng.mads_solve_batch(X0, 100, 1.0, 40)
    assert np.array_equal(res, X) and np.array_equal(objs, o) and runtime > 0
    assert st["batches"] == 1 and st["per_solve_iterations"] == s["iterations"].tolist()
    assert st["evaluations"] == s["evaluations"].sum() and st["best"] == int(np.argmin(o))
    res_py, objs_py, _ = OPT.optimize_multistart(X0, obj, [TC.cons1, cons3], [], 100, seed=40)  # default: Python
    assert res_py.shape == res.shape and np.isfinite(objs_py).sum() == np.isfinite(objs).sum()
    with pytest.raises(ValueError):
        OPT.optimize_multistart(X0, obj, [TC.cons1, cons3, lambda x: True], [], 5, native=True)
    with pytest.raises(ValueError):
        OPT.optimize_multistart(X0, obj, [TC.cons1], [], 5, granularity=np.ones(3 * N), native=True)
    cells.close()
