"""The device solver's own evaluator (mads_eval, cov_mads.cu) against the C oracle, at every launch width.

cov_mads_solve_batch, the horizons and both ensembles evaluate candidates with mads_eval, not with the span kernels:
each warp paints the (disc, row) items of a candidate into its own framebuffer in shared memory (or replays the list
order for non-dyadic weights).  mads_plan picks W = 8, 4, 2 or 1 warps per CTA, halving until W framebuffers fit,
and stages the bit planes in shared memory when they fit beside them (mads_kernel<MULTI, PLANES_SMEM>).

The probe: cov_mads_solve_batch with n_iter = 0 evaluates X0[k] alone, on warp 0 of a CTA, and returns X0[k], its
barrier value and stats [0, 1, 0, 0].  So any candidate set goes through the solver's evaluator, and its value must
equal the oracle's barrier value (obj where feasible and obj == obj, else +Inf) bit for bit.

CPU: the kernels nvcc built are exactly the rows of SOLVER_VARIANTS; mads_plan restated in Python lands every lab
grid on the (W, PLANES_SMEM) row the PLAN_TABLE claims, and the lab reaches all 16 (W, PLANES_SMEM, MULTI) rows.
W = 1 is not always L2: at 1024 x 875 one framebuffer and one plane both fit, and mads_kernel<*, 1> runs with one
warp.  MULTI = 1 with one plane (one class, every multiplicity 2) reaches the shared-memory rows at W = 2 and 1.

GPU: the probe against the oracle on every table row, N = 1 .. 64, COV_OPT_FORCE_EXACT 0 and 1: edge-value swarms
without constraints (so that every one of them is painted), random, band-edge and near-boundary candidates with
cons3, cons7 and cons8 on for half of them; the list-order path; whole solves
against the host model of test_mads_device on every (W, PLANES_SMEM, MULTI) row, with exact radicand ties in the
poll points of every warp; the scenario kernels on W = 1 and W = 2 grids; the region solver's evaluator; the largest
grid the library accepts at the W = 1 boundary against the restatement."""
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from test_launch_matrix import _band_candidates, _candidates, _near_boundary_discs
from test_mads_device import assert_same, model_batch

T = math.tan((100 / 180 * math.pi) / 2)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "maximumareacoverageoptimization.jl_b200", "libcoverage_cuda.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
B200_OPTIN = 232448  # sharedMemPerBlockOptin of the B200 (227 KiB)
SEP = 15.0

# The solver's kernels and their template arguments: mads_kernel<MULTI, PLANES_SMEM, THREADS, CTAS>,
# scenario_solve_kernel<MULTI>, scenario_eval_kernel<MULTI>, region_solve_kernel<THREADS, CTAS>.
SOLVER_VARIANTS = {
    "mads_kernel": {(0, 0, 256, 2), (0, 1, 256, 2), (1, 0, 256, 2), (1, 1, 256, 2)},
    "scenario_solve_kernel": {(0,), (1,)},
    "scenario_eval_kernel": {(0,), (1,)},
    "region_solve_kernel": {(256, 2)},
}


# ---------------------------------------------------------------- mads_plan, restated
def _r16(v):
    return (v + 15) // 16 * 16


def mads_state_bytes(n):
    return _r16(7 * n * 8 + 2 * n * 4) + 64


def _stride(nx):
    return ((nx + 31) // 32) | 1  # words per row, rounded up to an odd count


def _plane_words(nx, ny):
    return (ny * _stride(nx) + 3) // 4 * 4


def mads_fb_bytes(nx, ny, N):
    return max(_r16(ny * _stride(nx) * 4), _r16(N * 8))  # the list-order path keeps N thresholds there


def mads_warp_bytes(nx, ny, N):
    return _r16(3 * N * 8) + N * 32 + _r16(N * 4) + mads_fb_bytes(nx, ny, N)


def mads_plan(nx, ny, n_planes, N, optin):
    """(warps per CTA, planes in shared memory), or None where the library refuses with COV_ERR_LIMIT."""
    if not 1 <= N <= 64:
        return None
    fixed, per_warp = mads_state_bytes(3 * N) + 16, mads_warp_bytes(nx, ny, N)
    w = 8
    while w > 1 and fixed + w * per_warp > optin:
        w //= 2
    if fixed + w * per_warp > optin:
        return None
    return w, n_planes * _plane_words(nx, ny) * 4 + fixed + w * per_warp <= optin


# (nx, ny, planes): (W, planes in shared memory) at N = 5 and the B200's opt-in shared memory; None: refused
PLAN_TABLE = {
    (256, 256, 1): (8, True), (256, 256, 2): (8, True), (256, 256, 8): (8, True),
    (400, 400, 1): (8, True), (400, 400, 2): (8, True), (400, 400, 8): (8, False),
    (512, 512, 1): (4, True), (512, 512, 2): (4, True), (512, 512, 8): (4, False),
    (600, 600, 1): (4, True), (600, 600, 2): (4, False),
    (700, 700, 1): (2, True), (700, 700, 2): (2, False),
    (800, 800, 1): (2, False), (800, 800, 2): (2, False),
    (1024, 1024, 1): (1, False), (1024, 1024, 2): (1, False), (32, 32768, 1): (1, False), (32, 32768, 2): (1, False),
    (33, 32768, 1): None, (8192, 8192, 1): None,
    # the rows the grids above leave out: one plane in L2 at W = 8 and 4, one plane in shared memory at W = 1
    (450, 450, 1): (8, False), (640, 640, 1): (4, False), (1024, 875, 1): (1, True), (420, 420, 2): (8, False),
    (512, 846, 2): (2, True),
}
ALL_ROWS = {(w, ps, multi) for w in (8, 4, 2, 1) for ps in (True, False) for multi in (0, 1)}


# ---------------------------------------------------------------- CPU
def _names():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    return set(re.findall(r"Function (\S+):", out))


@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_every_solver_instantiation_has_a_row():
    built = {k: set() for k in SOLVER_VARIANTS}
    for name in _names():
        m = re.search(r"cov(\d+)(mads_kernel|scenario_solve_kernel|scenario_eval_kernel|region_solve_kernel)I(\w+?)EEv",
                      name)
        if m:
            args = tuple(int(a) for a in re.findall(r"L[bi](\d+)E", m.group(3) + "E"))
            built[m.group(2)].add(args)
    assert built == SOLVER_VARIANTS, built
    assert sum(map(len, built.values())) == 4 + 2 + 2 + 1


def test_plan_restatement_table():
    for (nx, ny, planes), want in PLAN_TABLE.items():
        assert mads_plan(nx, ny, planes, 5, B200_OPTIN) == want, (nx, ny, planes, want)
    rows = {(w, ps) for w, ps in filter(None, PLAN_TABLE.values())}
    assert rows == {(w, ps) for w in (8, 4, 2, 1) for ps in (True, False)}
    # one warp's framebuffer is the limit: the largest accepted ny at nx = 1024 and N = 5
    assert mads_plan(1024, 1750, 1, 5, B200_OPTIN) == (1, False) and mads_plan(1024, 1751, 1, 5, B200_OPTIN) is None
    # the list-order path sizes a 4 x 4 grid's framebuffer by the N thresholds
    assert mads_fb_bytes(4, 4, 64) == 512 and mads_fb_bytes(4, 4, 5) == 48
    assert mads_plan(4, 4, 1, 64, B200_OPTIN) == (8, True) and mads_plan(1, 1, 1, 65, B200_OPTIN) is None
    # the lab below reaches every (W, PLANES_SMEM, MULTI) row, and each row of the host-model test is its own
    assert set(_rows_reached(B200_OPTIN)) == set(MODEL_ROWS) == ALL_ROWS
    for (w, ps, multi), name in MODEL_ROWS.items():
        nx, ny, _, _ = STORES[name]
        assert mads_plan(nx, ny, _planes(name), 5, B200_OPTIN) == (w, ps) and _multi(name) == multi, name


# ---------------------------------------------------------------- GPU: the lab
# name: (nx, ny, kind, d).  kind: "bits" one plane (set_grid_bits), "two" two weight classes of single entries
# (set_points: two planes), "eight" four classes with multiplicities up to 3 (set_grid_cells: eight planes), "double"
# one class with every multiplicity 0 or 2 (set_grid_cells: one plane of multiplicity 2, so MULTI = 1)
STORES = {
    "256_1": (256, 256, "bits", 1.0), "256_2": (256, 256, "two", 1.0), "256_8": (256, 256, "eight", 1.0),
    "400_8": (400, 400, "eight", 1.0), "420_2": (420, 420, "two", 1.0), "450_1": (450, 450, "bits", 1.0),
    "512_1": (512, 512, "bits", 1.0), "512_2": (512, 512, "two", 1.0), "512_8": (512, 512, "eight", 1.0),
    "600_2": (600, 600, "two", 1.0), "640_1": (640, 640, "bits", 1.0),
    "700_1": (700, 700, "bits", 1.0), "700_2": (700, 700, "two", 1.0), "800_1": (800, 800, "bits", 1.0),
    "1024_1": (1024, 1024, "bits", 1.0), "1024_2": (1024, 1024, "two", 1.0), "1024x875_1": (1024, 875, "bits", 1.0),
    "512x846_2": (512, 846, "two", 1.0), "700_m2": (700, 700, "double", 1.0), "1024x875_m2": (1024, 875, "double", 1.0),
    "tall": (32, 32768, "bits", 1.0), "band": (256, 107, "bits", 2.0), "wide": (1500, 23, "bits", 1.0),
    "1x1": (1, 1, "bits", 5.0), "4x4": (4, 4, "bits", 1.0),
}
NS = (1, 5, 31, 32, 33, 64)


def _build(cov, name):
    """(set-up function of an engine, the oracle's point list, n_planes) of a lab store."""
    nx, ny, kind, d = STORES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    ii, jj = np.meshgrid(np.arange(nx), np.arange(ny), indexing="ij")  # cell (i, j) at index i + nx j below
    if kind == "bits":
        fire = rng.random((nx, ny)) < (0.5 if nx * ny <= 16 else 0.12)
        fire[0, 0] = True
        if name == "tall":
            fire[:, -2:] = rng.random((nx, 2)) < 0.6  # rows 32767 and 32768
        bits = cov.synth.pack_bits(fire)
        pts = cov.synth.points_from_bits(bits, nx, d, d)
        return (lambda e: e.set_grid_bits(bits, nx, ny, d, d)), pts, 1
    if kind == "two":
        on = rng.random((nx, ny)) < 0.12
        pts = np.stack([(ii[on] + 0.5) * d, (jj[on] + 0.5) * d, np.full(on.sum(), d * d),
                        np.where(rng.random(on.sum()) < 0.5, 1.0, 2.0) * d * d, np.zeros(on.sum())], axis=1)
        pts = pts[rng.permutation(len(pts))]
        return (lambda e: e.set_points(pts, nx, ny, d, d)), pts, 2
    if kind == "double":
        mult = np.where(rng.random((nx, ny)) < 0.12, 2, 0).astype(np.uint8)
        rep = mult.ravel(order="F")
        pts = np.stack([np.repeat((ii.ravel(order="F") + 0.5) * d, rep), np.repeat((jj.ravel(order="F") + 0.5) * d, rep),
                        np.full(rep.sum(), d * d), np.full(rep.sum(), d * d), np.zeros(rep.sum())], axis=1)
        return (lambda e: e.set_grid_cells(rep, nx, ny, d, d)), pts, 1
    mult = np.where(rng.random((nx, ny)) < 0.12, rng.integers(1, 4, (nx, ny)), 0).astype(np.uint8)
    cls = rng.integers(0, 4, (nx, ny)).astype(np.uint8)
    cw = np.array([1.0, 2.0, 0.5, 4.0]) * d * d
    rep = mult.ravel(order="F")
    pts = np.stack([np.repeat((ii.ravel(order="F") + 0.5) * d, rep), np.repeat((jj.ravel(order="F") + 0.5) * d, rep),
                    np.full(rep.sum(), d * d), np.repeat(cw[cls.ravel(order="F")], rep), np.zeros(rep.sum())], axis=1)
    return (lambda e: e.set_grid_cells(mult.ravel(order="F"), nx, ny, d, d, cls=cls.ravel(order="F"),
                                       class_weight=cw)), pts, 8


def _edge_rows(N, cx, cy):
    """test_gpu_parity's edge-value swarms (R = 0, negative, NaN, +Inf, denormal, 1e300, 1e18 absorption, NaN / Inf
    centres) around (cx, cy), padded to N discs with small discs beside them."""
    inf, nan = math.inf, math.nan
    pairs = [((cx, cy, 0.0), (cx, cy, 0.0)), ((cx, cy, -5.0), (cx, cy, -0.0)), ((cx, cy, nan), (cx, cy, 10.0)),
             ((cx, cy, inf), (cx, cy, 1.0)), ((-1e6, cy, 30.0), (1e6, cy, 30.0)), ((1e300, 250, 1e300), (250, -1e300, 20.0)),
             ((cx, 1e18, 1e18), (cx, cy, 3.0)), ((0.5, 0.5, 2.5), (cx, cy, 2.6)), ((cx, cy, 1e-300), (cx, cy, 5e-324)),
             ((nan, cy, 10.0), (cx, cy, 10.0)), ((inf, cy, inf), (cx, cy, 10.0)), ((0.0, 0.0, 1e4), (cx, cy, 1.0))]
    rows = []
    for p in pairs:
        discs = list(p) if N > 1 else [p[0]]
        discs += [(cx - 40 + 2.5 * k, cy + 30, 4.0) for k in range(N - len(discs))]
        if N == 1:
            rows.append([p[1]])
        rows.append(discs[:N])
    X = np.array(rows)  # (B, N, 3)
    return np.concatenate([X[:, :, 0], X[:, :, 1], X[:, :, 2]], axis=1)


def _pool(name, N):
    nx, ny, _, d = STORES[name]
    rng = np.random.default_rng(1000 * N + sum(map(ord, name)))
    big = nx * ny >= 256 * 256
    B = {1: 2500, 5: 2000}.get(N, 200) if big else {1: 3000, 5: 2000}.get(N, 300)
    # the edge rows first, so that they fall in the half evaluated without constraints and reach the painting code
    parts = [_edge_rows(N, nx * d / 2, ny * d / 2), _candidates(rng, B, N, nx, ny, d)]
    nb = np.array(_near_boundary_discs(rng, max(B // 2, 8) * N, nx, ny, d)).reshape(-1, N, 3)
    parts.append(np.concatenate([nb[:, :, 0], nb[:, :, 1], nb[:, :, 2]], axis=1))
    if name == "band":  # N = 1: the discs of the 5-disc band candidates one by one
        X5 = _band_candidates(rng, 5 if N == 1 else N)[:B]
        parts.append(X5.reshape(-1, 3, 5).transpose(0, 2, 1).reshape(-1, 3) if N == 1 else X5)
    if name == "tall":  # discs on the last rows (the 16-bit row field of a disc's row range)
        top = _candidates(rng, B // 2, N, nx, 8, d)
        top[:, N:2 * N] += (ny - 8) * d
        parts.append(top)
    if name == "wide":  # chords across the grid
        w = _candidates(rng, B // 2, N, nx, ny, d)
        w[:, 2 * N:] = 200 + rng.random((B // 2, N)) * 700
        parts.append(w)
    return np.concatenate(parts)


def _params(engine, N, constrained, penalty=1e5, centre=(250.0, 250.0)):
    """Half the rows run with cons3 (d_lim 300-700 m around a swarm at centre), cons7 and cons8."""
    if not constrained:
        engine.set_params(N, np.full(N, 30 * T), penalty)
        return {}
    rng = np.random.default_rng(N)
    prev = np.concatenate([np.full(N, centre[0]), np.full(N, centre[1]), np.full(N, 20.0)])
    kw = dict(pre=prev, d_lim=rng.uniform(300, 700, N), tan_half_fov=T, sep_min=SEP, use_cons7=True)
    engine.set_params(N, np.full(N, 30 * T), penalty, prev_xyR=prev, d_lim=kw["d_lim"], tan_half_fov=T, sep_min=SEP,
                      use_cons7=True)
    return kw


def _barrier(r):
    return np.where((r["feasible"] != 0) & (r["obj"] == r["obj"]), r["obj"], math.inf)


def probe(engine, X):
    """mads_eval's barrier value of every row of X (cov_mads_solve_batch, n_iter = 0)."""
    Xo, obj, st = engine.mads_solve_batch(X, 0, 1.0, 0)
    assert np.array_equal(Xo.view(np.uint64), X.view(np.uint64))
    assert np.all(st["iterations"] == 0) and np.all(st["evaluations"] == 1)
    assert np.all(st["successes"] == 0) and np.all(st["converged"] == 0)
    return obj


def _bad(got, want):
    return np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))


def _optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


class Lab:
    def __init__(self, cov, orc):
        self.cov, self.orc, self.eng = cov, orc, cov.CoverageEngine(0)
        self.built, self.store = {}, None

    def set_store(self, name):
        if name not in self.built:
            self.built[name] = _build(self.cov, name)
        setup, pts, planes = self.built[name]
        if self.store != name:
            setup(self.eng)
            info = self.eng.grid_info()
            assert info["area_exact"] == 1 and info["n_planes"] == planes, (name, info)
            assert info["n_entries"] == len(pts), name
            self.store = name
        return pts

    def close(self):
        self.eng.close()


@pytest.fixture(scope="module")
def lab(cov, orc):
    lb = Lab(cov, orc)
    yield lb
    lb.close()


def _planes(name):
    return {"bits": 1, "two": 2, "eight": 8, "double": 1}[STORES[name][2]]


def _multi(name):
    return int(STORES[name][2] != "bits")  # mads_kernel<MULTI = 1> unless one plane of one class, multiplicity 1


def _rows_reached(optin):
    """{(W, PLANES_SMEM, MULTI): [(store, N)]} of every probe of test_evaluator_against_the_oracle."""
    out = {}
    for name, (nx, ny, _, _) in STORES.items():
        for N in NS:
            p = mads_plan(nx, ny, _planes(name), N, optin)
            if p is not None:
                out.setdefault((p[0], p[1], _multi(name)), []).append((name, N))
    return out


# ---------------------------------------------------------------- GPU: the evaluator against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(STORES))
def test_evaluator_against_the_oracle(cov, orc, lab, name):
    optin, sms = _optin(), _sms()
    nx, ny, kind, d = STORES[name]
    planes = _planes(name)
    if (nx, ny, planes) in PLAN_TABLE:
        assert mads_plan(nx, ny, planes, 5, optin) == PLAN_TABLE[nx, ny, planes], (name, optin)
    compared, persistent, feasible, constrained_rows = 0, False, 0, 0
    centre = (nx * d / 2, ny * d / 2)
    for N in NS:
        if mads_plan(nx, ny, planes, N, optin) is None:
            continue
        pts = lab.set_store(name)
        X = _pool(name, N)
        h = len(X) // 2
        want = np.empty(len(X))
        for rows, constrained in ((slice(0, h), False), (slice(h, None), True)):
            kw = _params(lab.eng, N, constrained, centre=centre)
            r = orc.eval_batch(X[rows], N, np.full(N, 30 * T), pts, **kw)
            want[rows] = _barrier(r)
            if not constrained:
                ref = r
                ne = len(_edge_rows(N, 0.0, 0.0))  # edge rows: unconstrained, so all go through the painting code
                assert r["feasible"][:ne].all() and (r["count"][:ne] > 0).any(), (name, N)
            else:
                feasible += int(r["feasible"].sum())
                constrained_rows += len(r["feasible"])
            for fe in (0, 1):
                lab.eng.set_option(cov.OPT_FORCE_EXACT, fe)
                got = probe(lab.eng, X[rows])
                bad = _bad(got, want[rows])
                assert bad.size == 0, (name, N, constrained, fe, bad[:8], got[bad[:4]], want[rows][bad[:4]])
            lab.eng.set_option(cov.OPT_FORCE_EXACT, 0)
        if kind == "bits":  # penalty_scale = 0: -obj is the covered weight itself
            _params(lab.eng, N, False, penalty=0.0)
            w0 = np.where(np.isfinite(want[:h]), -(ref["count"] * (d * d)) + 0.0, math.inf)
            got = probe(lab.eng, X[:h])
            bad = _bad(got, w0)
            assert bad.size == 0, (name, N, "penalty 0", bad[:8], got[bad[:4]], w0[bad[:4]])
        compared += len(X)
        # more solves than CTAs can be resident (256-thread CTAs, at most 2048 threads per SM): persistent CTAs take
        # the later ones from the dispenser
        persistent |= h > 8 * sms
    assert compared > 0 and persistent
    assert 0 < feasible < constrained_rows, (name, feasible, constrained_rows)  # the barrier takes part
    print(f"\n{name}: {nx} x {ny}, {planes} plane(s), plan at N = 5 {mads_plan(nx, ny, planes, 5, optin)}: "
          f"{compared} candidates x 2 FORCE_EXACT compared, {feasible} of {constrained_rows} constrained rows feasible")


# ---------------------------------------------------------------- GPU: the list-order path
@pytest.mark.gpu
def test_list_order_path_against_the_oracle(cov, orc, engine):
    """Non-dyadic weights (area_exact == 0): mads_eval replays the reference's list-order Float64 sum."""
    rng = np.random.default_rng(77)
    total = 0
    for nx, d, Ns, Ps in ((100, 5.0, (1, 31, 32, 33, 64), (0, 1, 31, 32, 33, 3000)), (4, 5.0, (64,), (0, 1, 33, 3000))):
        for P in Ps:
            i, j = rng.integers(0, nx, P), rng.integers(0, nx, P)
            hi = (30 * T) ** 2 * math.pi  # the high-interest weight: not dyadic
            # one weight per cell; two classes where the multiplicities stay small, else one (at most 8 bit planes)
            cell_w = np.where(rng.random(nx * nx) < 0.5, hi, d * d) if P <= nx * nx else np.full(nx * nx, hi)
            w = cell_w[i + nx * j]
            pts = np.stack([(i + 0.5) * d, (j + 0.5) * d, np.full(P, d * d), w, np.zeros(P)], axis=1)
            engine.set_points(pts, nx, nx, d, d)
            exact = engine.grid_info()["area_exact"]
            assert exact == 0 or P < 2, (nx, P)
            for N in Ns:
                X = _candidates(rng, 300 if N < 32 else 120, N, nx, nx, d)
                X = np.concatenate([_edge_rows(N, nx * d / 2, nx * d / 2), X])  # edge rows in the unconstrained half
                h = len(X) // 2
                for rows, constrained in ((slice(0, h), False), (slice(h, None), True)):
                    kw = _params(engine, N, constrained)
                    want = _barrier(orc.eval_batch(X[rows], N, np.full(N, 30 * T), pts, **kw))
                    for fe in (0, 1):
                        engine.set_option(cov.OPT_FORCE_EXACT, fe)
                        got = probe(engine, X[rows])
                        bad = _bad(got, want)
                        assert bad.size == 0, (nx, P, N, constrained, fe, bad[:8], got[bad[:4]], want[bad[:4]])
                    engine.set_option(cov.OPT_FORCE_EXACT, 0)
                total += len(X)
    print(f"\nlist order: {total} candidates compared")


# ---------------------------------------------------------------- GPU: whole solves on every launch row
MODEL_ROWS = {  # (W, PLANES_SMEM, MULTI): lab store, every one of ALL_ROWS
    (8, True, 0): "256_1", (8, False, 0): "450_1", (4, True, 0): "512_1", (4, False, 0): "640_1",
    (2, True, 0): "700_1", (2, False, 0): "800_1", (1, True, 0): "1024x875_1", (1, False, 0): "1024_1",
    (8, True, 1): "256_2", (8, False, 1): "400_8", (4, True, 1): "512_2", (4, False, 1): "512_8",
    (2, True, 1): "700_m2", (2, False, 1): "700_2", (1, True, 1): "1024x875_m2", (1, False, 1): "1024_2",
}


@pytest.mark.gpu
@pytest.mark.parametrize("row", list(MODEL_ROWS), ids=lambda r: "w%d-%s-multi%d" % (r[0], "smem" if r[1] else "l2", r[2]))
def test_solves_against_the_host_model(cov, lab, row):
    """mads_kernel's whole loop on every (W, PLANES_SMEM, MULTI) row against test_mads_device's host model.  Centres
    and radii on the 0.5 mesh of granularity 0.5, cells of pitch 1 on every store of MODEL_ROWS: poll points of every warp meet cells whose
    radicand equals T(R) exactly (Pythagorean offsets)."""
    name = MODEL_ROWS[row]
    nx, ny, _, d = STORES[name]
    N, n_iter, g, seed = 5, 14, 0.5, 2**64 - 3
    assert mads_plan(nx, ny, _planes(name), N, _optin()) == row[:2] and _multi(name) == row[2]
    lab.set_store(name)
    lab.eng.set_params(N, np.full(N, 30 * T), sep_min=SEP)
    rng = np.random.default_rng(sum(map(ord, name)) + 5)
    S = 4 if nx * ny > 300 * 300 else 8
    cx, cy = rng.uniform(0.3, 0.7, 2) * (nx * d, ny * d)
    X0 = np.concatenate([np.rint((cx + rng.uniform(-60, 60, (S, N))) / g) * g,
                         np.rint((cy + rng.uniform(-60, 60, (S, N))) / g) * g,
                         rng.choice([5.0, 10.0, 12.5, 13.0, 15.0, 17.0, 25.0], (S, N))], axis=1)
    got = lab.eng.mads_solve_batch(X0, n_iter, g, seed)
    want = model_batch(cov.synth, lab.eng, X0, n_iter, g, seed)
    assert_same(got, want)
    assert got[2]["successes"].sum() > 0 and got[2]["iterations"].min() > 1


@pytest.mark.gpu
def test_every_launch_row_is_reached():
    """With this device's opt-in shared memory, the stores and swarm sizes of test_evaluator_against_the_oracle put
    mads_kernel on every (W, PLANES_SMEM, MULTI) row, as test_solves_against_the_host_model does."""
    optin = _optin()
    reached = _rows_reached(optin)
    assert set(reached) == set(MODEL_ROWS), (optin, sorted(set(MODEL_ROWS) - set(reached)))
    for row in sorted(reached, reverse=True):
        print("\nW = %d, planes in %s, MULTI = %d (optin %d bytes):" % (row[0], "shared memory" if row[1] else "L2",
                                                                     row[2], optin), reached[row])


# ---------------------------------------------------------------- GPU: the W = 1 boundary
@pytest.mark.gpu
def test_largest_accepted_grid_equals_the_restatement(cov, engine):
    """At nx = 1024 and N = 5 the library accepts exactly the heights the restatement gives a plan."""
    optin = _optin()
    engine.set_grid_full(100, 100, 5.0, 5.0)
    engine.set_params(5, np.full(5, 30 * T))
    X = np.concatenate([np.full(10, 50.0), np.full(5, 10.0)])[None]

    def accepted(ny):
        engine.set_grid_full(1024, ny, 0.5, 0.5)
        try:
            probe(engine, X)
            return True
        except cov.CoverageError as e:
            assert e.code == cov._lib.COV_ERR_LIMIT, (ny, e)  # a refusal, never a failed launch
            return False

    lo, hi = 1, 32768  # accepted(lo), not accepted(hi)
    assert accepted(lo) and not accepted(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if accepted(mid) else (lo, mid)
    want = max(ny for ny in range(1, 4096) if mads_plan(1024, ny, 1, 5, optin) is not None)
    print(f"\nlargest accepted ny at nx = 1024, N = 5: {lo} (restatement {want}, optin {optin} bytes)")
    assert lo == want
    assert accepted(want) and mads_plan(1024, want, 1, 5, optin)[0] == 1


# ---------------------------------------------------------------- GPU: the scenario kernels off W = 8
@pytest.mark.gpu
def test_horizon_ensemble_on_one_warp(cov, engine):
    """scenario_solve_kernel / scenario_eval_kernel with W = 1 (1024 x 1024): every scenario equals cov_run_horizon."""
    from test_horizon_ensemble import STAT_NAMES, _bits
    N, E, T_, S = 5, 3, 3, 2
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    assert mads_plan(1024, 1024, 1, N, _optin())[0] == 1

    def prep(eng):
        eng.set_grid_full(1024, 1024, 0.5, 0.5)
        eng.set_params(N, np.full(N, 30 * T), 1e5, prev_xyR=x0, d_lim=10.0, tan_half_fov=T)

    prep(engine)
    starts = np.repeat(x0[None], E, axis=0)
    starts[1:, :2 * N] += np.rint(np.random.default_rng(4).uniform(-30, 30, (E - 1, 2 * N)))
    kw = dict(T=T_, S=S, n_iter=10, granularity=1.0, seed=2**64 - 11)
    X, obj, st, _, cells = engine.run_horizon_ensemble(starts, want_cells=True, **kw)
    ref = cov.CoverageEngine(0)
    try:
        for e in range(E):
            prep(ref)
            Xr, objr, str_, _ = ref.run_horizon(starts[e], **dict(kw, seed=(kw["seed"] + e * T_ * S) % 2**64))
            assert np.array_equal(_bits(X[e]), _bits(Xr)) and np.array_equal(_bits(obj[e]), _bits(objr)), e
            for k in STAT_NAMES:
                assert np.array_equal(st[k][e], str_[k]), (e, k)
            assert np.array_equal(cells[e], ref.grid_cells()), e  # the store each scenario leaves
    finally:
        ref.close()
    assert st["removed"].sum() > 0


@pytest.mark.gpu
def test_fire_ensemble_on_two_warps(cov, engine):
    """The fire ensemble with W = 2 (an 800 x 800 fire of pitch 0.625): every scenario equals cov_run_horizon_fire."""
    from test_horizon_fire_ensemble import STAT_NAMES, _bits
    N, E, S = 5, 2, 2
    fs = np.array([0, 1, 1], dtype=np.int64)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 330.0)
    assert mads_plan(800, 800, 1, N, _optin())[0] == 2
    wind = (4.0, math.radians(270.0), 0.5)

    def prep(eng):
        ff = cov.DynamicArea.ForestFire(eng, dx=0.625, dy=0.625, seed=3)
        eng.set_params(N, np.full(N, 30 * T), 1e5, prev_xyR=x0, d_lim=10.0, tan_half_fov=T)
        return ff

    ff = prep(engine)
    starts = np.repeat(x0[None], E, axis=0)
    starts[1:, :2 * N] += np.rint(np.random.default_rng(5).uniform(-40, 40, (E - 1, 2 * N)))
    kw = dict(S=S, n_iter=10, granularity=1.0, seed=2**64 - 13)
    X, obj, st, _, cells, states = ff.run_horizon_ensemble(starts, fs, np.repeat(np.array([wind]), E, axis=0),
                                                           want_cells=True, want_states=True, **kw)
    ref = cov.CoverageEngine(0)
    try:
        for e in range(E):
            rf = prep(ref)
            Xr, objr, str_, _ = ref.run_horizon_fire(starts[e], fs, *wind, (rf.seed + e) % 2**64, rf.t + 1,
                                                     **dict(kw, seed=(kw["seed"] + e * len(fs) * S) % 2**64))
            assert np.array_equal(_bits(X[e]), _bits(Xr)) and np.array_equal(_bits(obj[e]), _bits(objr)), e
            for k in STAT_NAMES:
                assert np.array_equal(st[k][e], str_[k]), (e, k)
            assert np.array_equal(cells[e], ref.grid_cells()), e     # the store each scenario leaves
            assert np.array_equal(states[e], ref.fire_state()), e    # and its automaton state
    finally:
        ref.close()
    assert st["appended"].sum() > 0 and st["removed"].sum() > 0


# ---------------------------------------------------------------- GPU: the region solver's evaluator
@pytest.mark.gpu
def test_region_solver_evaluator(cov, engine):
    """cov_mads_solve_batch_region with n_iter = 0 returns cov_eval_region_batch's barrier value bit for bit; at
    M = 512 (the most covered discs) the area also matches the slab restatement."""
    import test_region_objective as tro
    rng = np.random.default_rng(512)
    total = 0
    for M in (0, 1, 200, 512):
        C3 = tro._covered_set(rng, M)
        if M == 512:
            C3[:, 2] *= 0.5  # smaller discs: the boundary's arcs stay within what the kernels take
        engine.set_region(*tro.DOMAIN, C3)
        for N, B in ((1, 600), (5, 400), (17, 120), (64, 24)):
            X = tro._candidates(rng, B, N, C3)
            tro._params(engine, N, rng)
            ev = engine.eval_region_batch(X)
            want = _barrier(ev)
            Xo, obj, st = engine.mads_solve_batch_region(X, 0, 1.0, 0)
            assert np.array_equal(Xo.view(np.uint64), X.view(np.uint64)) and np.all(st["evaluations"] == 1)
            bad = _bad(obj, want)
            assert bad.size == 0, (M, N, bad[:8], obj[bad[:4]], want[bad[:4]])
            if M == 512 and N in (1, 5):
                ref = tro.ref_batch(X[:150], N, C3)
                bad = np.abs(ev["area"][:150] - ref) > np.maximum(1e-9 * np.abs(ref), tro.ATOL)
                assert not bad.any(), (N, np.flatnonzero(bad)[:5], ev["area"][:150][bad][:5], ref[bad][:5])
            total += B
    print(f"\nregion: {total} candidates compared")
