"""The grid-free static objective (cov_set_region / cov_eval_region_batch / cov_mads_solve_batch_region).

A(x) = |(D_1 u ... u D_N) n Omega \\ C| is restated here independently of the kernels' boundary integration: by slabs.
For each y the covered x-length of the region is |U(D u C) n [x_lo, x_hi]| - |U(C) n [x_lo, x_hi]| (a union of
intervals less a union of intervals), integrated over y with adaptive Gauss-Legendre between the y-breakpoints (circle
tops and bottoms, pairwise circle intersections, circle / side-edge intersections).  CPU: the restatement against
closed forms; what nvcc built for the new kernels.  GPU: the kernels against the restatement, the grid objective's
convergence to A(x), the objective assembly and poll winner, determinism, the device MADS against a host model, and
the Python surface."""
import math
import os
import re
import shutil
import subprocess
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

T = math.tan((100 / 180 * math.pi) / 2)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "maximumareacoverageoptimization.jl_b200", "libcoverage_cuda.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
DOMAIN = (0.0, 0.0, 500.0, 500.0)
ATOL = 1e-9 * 500.0 * 500.0  # 1e-9 of the domain's area

# ---------------------------------------------------------------- the restatement
_GL = {n: np.polynomial.legendre.leggauss(n) for n in (12, 24)}


def _union_length(a, b):
    """Row-wise measure of the union of the intervals [a, b] (K x P; empty ones have b <= a)."""
    order = np.argsort(a, axis=1)
    a = np.take_along_axis(a, order, 1)
    b = np.take_along_axis(b, order, 1)
    prev = np.maximum.accumulate(b, axis=1)
    prev = np.concatenate([np.full((len(a), 1), -np.inf), prev[:, :-1]], axis=1)
    return np.clip(b - np.maximum(a, prev), 0.0, None).sum(axis=1)


def _chords(y, discs, x_lo, x_hi):
    """x-intervals of the discs (P x 3 rows x, y, R) at the heights y (K), clipped to [x_lo, x_hi]."""
    dy = y[:, None] - discs[None, :, 1]
    h2 = discs[None, :, 2] ** 2 - dy * dy
    w = np.sqrt(np.where(h2 > 0, h2, 0.0))
    a = np.clip(discs[None, :, 0] - w, x_lo, x_hi)
    b = np.clip(discs[None, :, 0] + w, x_lo, x_hi)
    return np.where(h2 > 0, a, x_lo), np.where(h2 > 0, b, x_lo)


def _length(y, D, Cv, x_lo, x_hi):
    aD, bD = _chords(y, D, x_lo, x_hi)
    if len(Cv) == 0:
        return _union_length(aD, bD)
    aC, bC = _chords(y, Cv, x_lo, x_hi)
    return _union_length(np.concatenate([aD, aC], 1), np.concatenate([bD, bC], 1)) - _union_length(aC, bC)


def _breakpoints(circ, x_lo, x_hi):
    ys = [circ[:, 1] - circ[:, 2], circ[:, 1] + circ[:, 2]]
    for xe in (x_lo, x_hi):  # circle / side-edge intersections
        h2 = circ[:, 2] ** 2 - (xe - circ[:, 0]) ** 2
        ok = h2 > 0
        ys += [circ[ok, 1] - np.sqrt(h2[ok]), circ[ok, 1] + np.sqrt(h2[ok])]
    i, j = np.triu_indices(len(circ), 1)
    c1, c2 = circ[i], circ[j]
    d = np.hypot(c2[:, 0] - c1[:, 0], c2[:, 1] - c1[:, 1])
    ok = (d < c1[:, 2] + c2[:, 2]) & (d > np.abs(c1[:, 2] - c2[:, 2]))
    c1, c2, d = c1[ok], c2[ok], d[ok]
    a = (c1[:, 2] ** 2 - c2[:, 2] ** 2 + d * d) / (2 * d)
    h = np.sqrt(np.clip(c1[:, 2] ** 2 - a * a, 0, None))
    py = c1[:, 1] + a * (c2[:, 1] - c1[:, 1]) / d
    off = h * (c2[:, 0] - c1[:, 0]) / d
    ys += [py - off, py + off]
    return np.concatenate(ys)


def _integrate(f, a, b, depth=0):
    """Adaptive Gauss-Legendre of f over [a, b] after y = a + (b - a)(3u^2 - 2u^3), which smooths the square-root
    ends of the chord lengths at circle tops and bottoms."""
    out = []
    for n in (12, 24):
        u, w = _GL[n]
        u = 0.5 * (u + 1.0)
        y = a + (b - a) * (3 * u * u - 2 * u ** 3)
        out.append(0.5 * (b - a) * np.sum(w * 6 * u * (1 - u) * f(y)))
    if abs(out[1] - out[0]) <= 1e-12 * max(1.0, (b - a) * 1000.0) or depth > 30:
        return out[1]
    m = 0.5 * (a + b)
    return _integrate(f, a, m, depth + 1) + _integrate(f, m, b, depth + 1)


def region_area_ref(x, N, covered=None, domain=DOMAIN):
    """A(x) by slab integration (float64 NumPy; shares nothing with the kernels)."""
    x_lo, y_lo, x_hi, y_hi = domain
    D = np.asarray(x, dtype=np.float64).reshape(3, N).T
    D = D[D[:, 2] > 0]
    C3 = np.zeros((0, 3)) if covered is None else np.asarray(covered, dtype=np.float64).reshape(-1, 3)
    C3 = C3[C3[:, 2] > 0]
    if not len(D):
        return 0.0
    # covered discs that meet no candidate disc remove nothing
    dd = np.hypot(C3[:, None, 0] - D[None, :, 0], C3[:, None, 1] - D[None, :, 1])
    Cv = C3[(dd < C3[:, None, 2] + D[None, :, 2]).any(axis=1)] if len(C3) else C3
    lo = max(y_lo, (D[:, 1] - D[:, 2]).min())
    hi = min(y_hi, (D[:, 1] + D[:, 2]).max())
    if not lo < hi:
        return 0.0
    br = _breakpoints(np.concatenate([D, Cv]), x_lo, x_hi)
    br = np.unique(np.concatenate([[lo, hi], br[(br > lo) & (br < hi)]]))
    f = lambda y: _length(y, D, Cv, x_lo, x_hi)  # noqa: E731
    return float(sum(_integrate(f, br[k], br[k + 1]) for k in range(len(br) - 1)))


def _ref_many(args):
    X, N, covered = args
    return [region_area_ref(x, N, covered) for x in X]


def ref_batch(X, N, covered):
    """region_area_ref over the rows of X, spread over the host's cores."""
    parts = np.array_split(X, max(1, min(len(X), 4 * (os.cpu_count() or 1))))
    with ProcessPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
        return np.array([a for part in ex.map(_ref_many, [(p, N, covered) for p in parts]) for a in part])


# ---------------------------------------------------------------- CPU: the restatement against closed forms
def _lens(R1, R2, d):
    a1 = R1 * R1 * math.acos((d * d + R1 * R1 - R2 * R2) / (2 * d * R1))
    a2 = R2 * R2 * math.acos((d * d + R2 * R2 - R1 * R1) / (2 * d * R2))
    return a1 + a2 - 0.5 * math.sqrt((-d + R1 + R2) * (d + R1 - R2) * (d - R1 + R2) * (d + R1 + R2))


def _close(got, want):
    assert abs(got - want) <= max(1e-9 * abs(want), 1e-9), (got, want)


def test_restatement_closed_forms():
    R, r = 30.0, 12.0
    _close(region_area_ref([250, 250, R], 1), math.pi * R * R)                        # inside
    _close(region_area_ref([250, 0, R], 1), math.pi * R * R / 2)                      # centred on an edge
    _close(region_area_ref([500, 250, R], 1), math.pi * R * R / 2)
    _close(region_area_ref([0, 0, R], 1), math.pi * R * R / 4)                        # centred on a corner
    _close(region_area_ref([500, 500, R], 1), math.pi * R * R / 4)
    _close(region_area_ref([250, 250, R], 1, [[240, 250, 45]]), 0.0)                  # inside C
    _close(region_area_ref([250, 250, R], 1, [[250, 250, R]]), 0.0)                   # identical to a covered disc
    _close(region_area_ref([250, 250, R], 1, [[250, 250, r]]), math.pi * (R * R - r * r))  # concentric hole
    _close(region_area_ref([250, 250, R], 1, [[250 + R - r, 250, r]]), math.pi * (R * R - r * r))  # internally tangent
    _close(region_area_ref([200, 230, 250, 250, R, r], 2), math.pi * (R * R + r * r) - _lens(R, r, 30.0))  # two discs
    _close(region_area_ref([200, 250, R], 1, [[230, 250, r]]), math.pi * R * R - _lens(R, r, 30.0))  # lens removed
    _close(region_area_ref([R, 250, R], 1), math.pi * R * R)                          # tangent to an edge
    _close(region_area_ref([250, 500 - R, R], 1), math.pi * R * R)
    _close(region_area_ref([250, 250, 250, 250, R, R], 2), math.pi * R * R)           # duplicate candidate discs
    _close(region_area_ref([-100, 250, R], 1), 0.0)                                   # outside the domain
    _close(region_area_ref([250, 250, 0.0], 1), 0.0)                                  # R = 0
    _close(region_area_ref([250, 250, 1000.0], 1), 500.0 * 500.0)                     # the whole domain


# ---------------------------------------------------------------- CPU: the compiled kernels
@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_region_kernels_fit_their_launch_plans():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    region = {k: v for k, v in usage.items() if "region_" in k}
    assert {re.search(r"region_\w+?_kernel", k).group(0) for k in region} == {
        "region_arcs_kernel", "region_eval_kernel", "region_solve_kernel"}, sorted(region)
    for k, v in region.items():
        assert v["LOCAL"] == 0 and v["STACK"] <= 128, (k, v)
        m = re.search(r"ILi(\d+)ELi(\d+)E", k)  # region_eval_kernel / region_solve_kernel<THREADS, CTAS>
        threads, ctas = map(int, m.groups()) if m else (32, 1)
        assert v["REG"] * threads * ctas <= 65536, (k, v)


# ---------------------------------------------------------------- GPU helpers
def _covered_set(rng, M):
    """M discs like the swarms of earlier timesteps: 5-disc rings at random centres, R ~ U(5, 35)."""
    out = []
    while len(out) < M:
        cx, cy, R = rng.uniform(0, 500), rng.uniform(0, 500), rng.uniform(5, 35)
        for i in range(5):
            a = 2 * math.pi * i / 5
            out.append([cx + 15 * math.cos(a), cy + 15 * math.sin(a), R * rng.uniform(0.8, 1.2)])
    return np.array(out[:M])


def _candidates(rng, B, N, C3):
    X = np.concatenate([rng.uniform(-40, 540, (B, 2 * N)), rng.uniform(0, 45, (B, N))], axis=1)
    X[:, 2 * N:][rng.random((B, N)) < 0.03] = 0.0
    for b in range(0, B, 3):  # adversarial discs in a third of the candidates
        i = rng.integers(N)
        R = rng.uniform(5, 40)
        kind = rng.integers(8)
        if kind == 0:
            d = [R, rng.uniform(0, 500), R]                              # tangent to the left edge
        elif kind == 1:
            d = [rng.uniform(0, 500), 500 - R, R]                        # tangent to the top edge
        elif kind == 2:
            d = [500.0 * rng.integers(2), 500.0 * rng.integers(2), R]    # centred on a corner
        elif kind == 3 and len(C3):
            d = list(C3[rng.integers(len(C3))])                          # identical to a covered disc
        elif kind == 4 and len(C3):
            cm = C3[rng.integers(len(C3))]                               # internally tangent to a covered disc
            r = cm[2] * rng.uniform(0.2, 0.9)
            a = rng.uniform(0, 2 * math.pi)
            d = [cm[0] + (cm[2] - r) * math.cos(a), cm[1] + (cm[2] - r) * math.sin(a), r]
        elif kind == 5:
            d = [-1000.0, 2000.0, R]                                     # far outside
        elif kind == 6 and N > 1:
            j = (i + 1) % N                                              # duplicate candidate discs
            d = [X[b, j], X[b, N + j], X[b, 2 * N + j]]
        else:
            d = [rng.uniform(0, 500), 0.0, R]                            # centred on an edge
        X[b, i], X[b, N + i], X[b, 2 * N + i] = d
    return X


def _params(engine, N, rng):
    """Parameters with every constraint on: cons3 around a swarm in the middle of the domain, cons7, cons8."""
    prev = np.concatenate([np.full(2 * N, 250.0), np.full(N, 20.0)])
    engine.set_params(N, np.full(N, 30 * T), prev_xyR=prev, d_lim=rng.uniform(300, 700, N), tan_half_fov=T, sep_min=15.0,
                      use_cons7=True)


# ---------------------------------------------------------------- GPU: the kernels against the restatement
CASES = [(N, M, B) for M in (0, 1, 40, 200) for N, B in ((1, 1200), (2, 700), (5, 500), (17, 90), (64, 12))]


@pytest.mark.gpu
def test_area_against_restatement(cov, engine):
    rng = np.random.default_rng(2024)
    total = 0
    for N, M, B in CASES:
        C3 = _covered_set(rng, M)
        X = _candidates(rng, B, N, C3)
        engine.set_region(*DOMAIN, C3)
        _params(engine, N, rng)
        got = engine.eval_region_batch(X)
        want = ref_batch(X, N, C3)
        err = np.abs(got["area"] - want)
        bad = err > np.maximum(1e-9 * np.abs(want), ATOL)
        assert not bad.any(), (N, M, np.flatnonzero(bad)[:5], got["area"][bad][:5], want[bad][:5])
        # the fused constraints are cov_eval_batch's, bit for bit
        engine.set_grid_full(100, 100, 5.0, 5.0)
        assert np.array_equal(got["feasible"], engine.eval_batch(X)["feasible"]), (N, M)
        assert 0 < got["feasible"].sum() < B or N > 5
        total += B
    assert total >= 10000


# ---------------------------------------------------------------- GPU: the limit the objective is defined by
@pytest.mark.gpu
def test_grid_objective_converges_to_region_area(cov, engine):
    """Config 1's setting: swarms t = 1..5 of allocate_even_circles, each earlier swarm removed from a createPOI store
    (cov_remove_covered) / added to the covered set.  |grid area - A| <= (boundary length) x (cell diagonal) at every
    dx = 500 / 2^k, k = 8..12, so the error shrinks at least like dx."""
    N = 5
    swarms = [cov.Base_Functions.allocate_even_circles(15.0, N, (10 + 3 * t) * T, 200.0 + 20 * t, 250.0 + 7 * t)
              for t in range(1, 6)]
    engine.set_params(N, swarms[0][2 * N:])
    A, bound = [], []
    for t, x in enumerate(swarms):
        C3 = np.concatenate([s.reshape(3, N).T for s in swarms[:t]]) if t else np.zeros((0, 3))
        engine.set_params(N, x[2 * N:])
        engine.set_region(*DOMAIN, C3)
        A.append(engine.eval_region_batch(x[None, :])["area"][0])
        assert abs(A[-1] - region_area_ref(x, N, C3)) <= 1e-9 * A[-1]
        D = x.reshape(3, N).T
        meets = [c for c in C3 if (np.hypot(D[:, 0] - c[0], D[:, 1] - c[1]) < D[:, 2] + c[2]).any()]
        bound.append(2 * math.pi * (D[:, 2].sum() + sum(c[2] for c in meets)))  # >= the boundary's length
    errs = {}
    for k in range(8, 13):
        n = 2 ** k
        dx = 500.0 / n
        engine.set_grid_full(n, n, dx, dx)
        for t, x in enumerate(swarms):
            engine.set_params(N, x[2 * N:])  # r_max = R: no penalty, obj = -count dx^2
            grid_area = -engine.eval_batch(x[None, :])["obj"][0]
            errs[k, t] = abs(grid_area - A[t])
            assert errs[k, t] <= bound[t] * dx * math.sqrt(2), (k, t, errs[k, t], bound[t] * dx * math.sqrt(2))
            engine.remove_covered(x)
    assert sum(errs[12, t] for t in range(5)) < sum(errs[8, t] for t in range(5)), errs  # and in fact it does shrink


# ---------------------------------------------------------------- GPU: objective assembly and the poll winner
@pytest.mark.gpu
def test_objective_assembly_and_winner(cov, engine):
    rng = np.random.default_rng(7)
    N = 5
    C3 = _covered_set(rng, 40)
    X = _candidates(rng, 600, N, C3)
    engine.set_region(*DOMAIN, C3)
    _params(engine, N, rng)
    r_max = np.full(N, 30 * T)
    got = engine.eval_region_batch(X)
    want_area = ref_batch(X, N, C3)
    assert np.allclose(got["area"], want_area, rtol=1e-9, atol=ATOL)
    for b in range(len(X)):  # -A + 1e5 * sum |R - r_max| in the grid objective's order, bit for bit
        viol = 0.0
        for i in range(N):
            viol += abs(X[b, 2 * N + i] - r_max[i])
        assert got["obj"][b] == -got["area"][b] + viol * 1e5
    assert 0 < got["feasible"].sum() < len(X)  # infeasible candidates keep their objective
    assert np.isfinite(got["obj"]).all()
    # the winner: cov_argmin's rule on ties (smallest index), with and without the barrier
    X2 = np.concatenate([X, X[::-1], X])
    for barrier in (True, False):
        res = engine.eval_region_batch(X2, best=True, barrier=barrier)
        f = np.where(res["feasible"] != 0, res["obj"], np.inf) if barrier else res["obj"]
        assert res["best"] == (f.min(), int(np.argmin(f)))
    # only infeasible candidates
    bad = X[got["feasible"] == 0]
    res = engine.eval_region_batch(bad, best=True)
    assert res["best"] == (math.inf, -1)
    assert engine.eval_region_batch(bad, best=True, barrier=False)["best"][1] == int(np.argmin(got["obj"][got["feasible"] == 0]))


@pytest.mark.gpu
def test_results_do_not_depend_on_the_batch(cov, engine):
    rng = np.random.default_rng(11)
    N = 5
    C3 = _covered_set(rng, 200)
    engine.set_region(*DOMAIN, C3)
    _params(engine, N, rng)
    X = _candidates(rng, 100000, N, C3)
    full = engine.eval_region_batch(X)
    again = engine.eval_region_batch(X)
    for key in ("obj", "area", "feasible"):
        assert np.array_equal(full[key].view(np.uint8), again[key].view(np.uint8)), key
    for B in (1, 7, 4096):
        for s in (0, 12345, 99999 - B):
            part = engine.eval_region_batch(X[s:s + B])
            for key in ("obj", "area", "feasible"):
                assert np.array_equal(part[key].view(np.uint8), full[key][s:s + B].view(np.uint8)), (B, s, key)


# ---------------------------------------------------------------- GPU: device MADS against the host model
def _model_batch(synth, eng, X0, n_iter, g, seed):
    from test_mads_device import _Model

    def barrier(P):
        if not len(P):
            return np.empty(0)
        r = eng.eval_region_batch(P, want_area=False)
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


def _c1_region(cov, engine, N=5, M=200, seed=1):
    """Config 1 on the region objective: the starting swarm, covered by M discs of earlier swarms."""
    rng = np.random.default_rng(seed)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    C3 = np.concatenate([_covered_set(rng, M - N), x0.reshape(3, N).T]) if M else np.zeros((0, 3))
    engine.set_region(*DOMAIN, C3)
    engine.set_params(N, np.full(N, 30 * T), prev_xyR=x0, d_lim=10.0, tan_half_fov=T)
    return x0


def _starts(rng, x0, S, N, spread=3.0, far=0):
    X0 = np.repeat(x0[None, :], S, axis=0)
    X0[:, :2 * N] += np.rint(rng.normal(0, spread, (S, 2 * N)))
    X0[:far, :N] += 60.0  # beyond cons3's 10 m: infeasible starts
    return X0


REGION_SCENARIOS = ["c1_cons3", "cons8", "gran_half", "gran_zero", "n1", "n64", "m0"]


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", REGION_SCENARIOS)
def test_mads_region_bit_for_bit_against_host_model(cov, engine, scenario):
    from test_mads_device import assert_same
    rng = np.random.default_rng(REGION_SCENARIOS.index(scenario) + 1)
    g, n_iter, seed, N = 1.0, 100, 23, 5
    if scenario == "n1":
        N = 1
    x0 = _c1_region(cov, engine, N, M=0 if scenario == "m0" else 200)
    X0 = _starts(rng, x0, 32 if scenario == "c1_cons3" else 8, N, far=4 if scenario == "c1_cons3" else 0)
    if scenario == "cons8":
        engine.set_params(N, np.full(N, 30 * T), sep_min=15.0)
        X0[:3, :N], X0[:3, N:2 * N] = 250.0 + np.arange(N) * 5.0, 300.0  # 5 m apart: these starts break cons8
    elif scenario == "gran_half":
        g = 0.5
    elif scenario == "gran_zero":
        g, n_iter = 0.0, 60
        X0 = X0 + rng.random(X0.shape) * 0.01
    elif scenario == "n64":
        N = 64
        engine.set_params(N, np.full(N, 20.0))
        X0 = np.concatenate([np.rint(rng.random((3, 2 * N)) * 500), np.rint(5 + rng.random((3, N)) * 20)], axis=1)
        n_iter = 8
    got = engine.mads_solve_batch_region(X0, n_iter, g, seed)
    want = _model_batch(cov.synth, engine, X0, n_iter, g, seed)
    assert_same(got, want)
    assert got[2]["iterations"].max() >= 1 and got[2]["successes"].sum() > 0
    if scenario in ("c1_cons3", "cons8"):
        assert np.any(~np.isfinite(_model_batch(cov.synth, engine, X0, 0, g, seed)[1]))


@pytest.mark.gpu
def test_mads_region_solves_are_independent(cov, engine):
    N = 5
    x0 = _c1_region(cov, engine, N)
    rng = np.random.default_rng(3)
    S, seed = 600, 2**64 - 100
    X0 = _starts(rng, x0, S, N, far=30)
    X, obj, st = engine.mads_solve_batch_region(X0, 100, 1.0, seed)
    for k in (0, 1, 99, 100, 377, 599):
        Xk, objk, stk = engine.mads_solve_batch_region(X0[k:k + 1], 100, 1.0, (seed + k) % 2**64)
        assert np.array_equal(Xk[0].view(np.uint64), X[k].view(np.uint64)) and objk[0] == obj[k]
        assert all(stk[name][0] == st[name][k] for name in st)


@pytest.mark.gpu
def test_region_errors_leave_the_handle_usable(cov, engine):
    L = cov._lib
    lib, h = L.lib, engine.handle
    X = np.full((2, 15), 100.0)
    out, obj = np.empty_like(X), np.empty(2)

    def ev(Xa=X, B=2, best=False):
        bo, bi = L.C.c_double(), L.C.c_int64()
        return lib.cov_eval_region_batch(h, Xa.ctypes.data, B, obj.ctypes.data, None, None, 1,
                                         L.C.byref(bo) if best else None, L.C.byref(bi) if best else None)

    def solve(S=2):
        return lib.cov_mads_solve_batch_region(h, X.ctypes.data, S, 5, 1.0, 0, out.ctypes.data, None, None)

    assert ev() == L.COV_ERR_STATE and solve() == L.COV_ERR_STATE  # nothing set
    engine.set_params(5, np.full(5, 30 * T))
    assert ev() == L.COV_ERR_STATE and solve() == L.COV_ERR_STATE  # no region (and never a grid)
    good = np.array([[100.0, 50.0, 20.0]])
    engine.set_region(*DOMAIN, good)
    assert ev() == L.COV_OK and solve() == L.COV_OK
    for args in ((0, 0, 0, 500), (0, 0, 500, -1), (math.nan, 0, 500, 500), (0, 0, math.inf, 500)):
        with pytest.raises(cov.CoverageError) as e:
            engine.set_region(*args)
        assert e.value.code == L.COV_ERR_INVALID
    with pytest.raises(cov.CoverageError) as e:
        engine.set_region(*DOMAIN, [[1.0, math.nan, 3.0]])
    assert e.value.code == L.COV_ERR_INVALID
    assert lib.cov_set_region(h, 0.0, 0.0, 500.0, 500.0, None, -1) == L.COV_ERR_INVALID
    with pytest.raises(cov.CoverageError) as e:
        engine.set_region(*DOMAIN, np.tile(good, (513, 1)))
    assert e.value.code == L.COV_ERR_LIMIT and "512" in e.value.message
    assert ev() == L.COV_OK  # the earlier region is still in place
    assert np.allclose(engine.eval_region_batch(X)["area"], region_area_ref(X[0], 5, good), rtol=1e-9)
    assert ev(best=True) == L.COV_OK and lib.cov_eval_region_batch(h, X.ctypes.data, 2, None, None, None, 1,
                                                                  L.C.byref(L.C.c_double()), None) == L.COV_ERR_INVALID
    assert ev(B=-1) == L.COV_ERR_INVALID and ev(B=0) == L.COV_OK and solve(S=-1) == L.COV_ERR_INVALID
    engine.set_params(65, np.full(65, 30 * T))
    with pytest.raises(cov.CoverageError) as e:
        engine.eval_region_batch(np.zeros((1, 195)))
    assert e.value.code == L.COV_ERR_LIMIT and "64" in e.value.message
    with pytest.raises(cov.CoverageError) as e:
        engine.mads_solve_batch_region(np.zeros((1, 195)), 5)
    assert e.value.code == L.COV_ERR_LIMIT and "64" in e.value.message
    engine.set_params(5, np.full(5, 30 * T))
    assert engine.mads_solve_batch_region(X, 5)[1].shape == (2,)
    engine.set_grid_full(100, 100, 5.0, 5.0)  # the cell store and the region do not touch each other
    assert np.isfinite(engine.eval_batch(X)["obj"]).all() and ev() == L.COV_OK


# ---------------------------------------------------------------- GPU: the Python surface
@pytest.mark.gpu
def test_optimize_multistart_native_on_the_region(cov):
    OPT, TC, ACC = cov.TDM_STATIC_opt, cov.TDM_Constraints, cov.AreaCoverageCalculation
    N, FOV = 5, 100 / 180 * math.pi
    r_max = np.full(N, 30.0 * T)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    obj = OPT.createRegionObjective(DOMAIN, x0.reshape(3, N).T, N, r_max)
    cons3 = TC.create_cons3(ACC.make_circles(x0), FOV, 10 * np.ones(N))
    X0 = _starts(np.random.default_rng(9), x0, 12, N)
    res, objs, runtime, st = OPT.optimize_multistart(X0, obj, [TC.cons1, cons3], [], 100, seed=40, return_stats=True,
                                                     native=True)
    X, o, s = obj._engine()[1].mads_solve_batch_region(X0, 100, 1.0, 40)
    assert np.array_equal(res, X) and np.array_equal(objs, o) and st["batches"] == 1
    assert np.isfinite(o).all()
    assert obj(res[0]) == o[0]
    xo, _ = OPT.optimize(x0, obj, [TC.cons1, cons3], [], 30, seed=1)  # the Python poll driver on .batch / .fuse
    assert obj(xo) <= obj(x0)
    obj.close()


@pytest.mark.gpu
def test_run_simulation_on_the_region(cov):
    CF, FS = cov.CellFunctions, cov.FullSimulation
    params = FS.SimulationParameters(seed=5, N_iter=30)
    cells = CF.initialise_POI(CF.Cells(), "static")
    N = params.N
    start = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    r_max = params.h_max * T * np.ones(N)
    covered = []
    inp, outp, runtimes, objs = FS.run_simulation(cells, start, cov.TDM_Constraints.cons1, [], N, r_max.copy(), params,
                                                  objective="region", covered_pb=covered)
    assert len(outp) == params.Nt_sim == 40 and len(covered) == 40
    for t in range(40):
        assert covered[t].shape == (N * (t + 1), 3)
        want = start if t == 0 else outp[t - 1]
        assert np.array_equal(covered[t][-N:], want.reshape(3, N).T)
    assert all(np.isfinite(o) for o in objs)
    with pytest.raises(ValueError):
        FS.run_simulation(cells, start, cov.TDM_Constraints.cons1, [], N, r_max, FS.SimulationParameters(
            environment_type="dynamic"), Nt_sim=1, objective="region")
    cells.close()
