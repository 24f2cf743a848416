"""The device kernels around the objective (cov_grid_kernels.cu) at their edges, each against an independent reference.

1. Poll winner (argmin_stage1/2 and the host merges of cov_argmin, cov_eval_batch_best, cov_eval_batch_packed and
   cov_multi_argmin): the winner is the smallest objective and, among equal objectives, the smallest index -- MADS's
   first strict minimum.  Duplicated rows give bit-identical objectives, so ties are placed on both sides of every
   layer that settles one: the warp, the CTA, stage 2, the grid-stride lap, the host window, the 4 MiB switch and
   the shard boundary.
2. Fire automaton (fire_step_kernel, fire_seed_kernel) against the C oracle driven by the same Philox stream, step
   by step, on non-square lattices, 64-bit seeds, extreme step counters, both flags and the overflow path; the CPU
   part checks the oracle against a NumPy transcription of update_grid.
3. Cell removal and covered mask (remove_covered_kernel, covered_mask_kernel) cell by cell against the reference
   predicate `sqrt(s) < R`, with radicands placed exactly on T(R) and one ulp either side.
4. Union area (union_area_kernel, union_area_big_kernel) against an mpmath reference that decides coverage by point
   tests at arc midpoints instead of merging angular intervals, so that a rule the kernels and the NumPy restatement
   share cannot hide an error."""
import ctypes as C
import math

import numpy as np
import pytest

T = math.tan((100 / 180 * math.pi) / 2)
EPS = 2.0 ** -52
gpu = pytest.mark.gpu


# ================================================================ 1. poll winner
# A 16 x 16 grid of unit cells, two UAVs at fixed centres; only the radii change, so the objective falls as the
# radii grow.  cons3 (previous radii 3, d_lim 1) admits radii 2..4 and rejects 1 and 5.  Every value is an integer,
# so the same rows go through the int16 packed entry unchanged.
PREV = np.array([4.0, 12.0, 8.0, 8.0, 3.0, 3.0])


def _row(r1, r2):
    return np.array([4.0, 12.0, 8.0, 8.0, float(r1), float(r2)])


BEST_FEASIBLE = _row(4, 4)    # the best feasible row
BEST_ANY = _row(5, 5)         # better still, but infeasible
FILLERS = np.array([_row(2, 2), _row(3, 3), _row(2, 3), _row(3, 2), _row(1, 1)])
LAP = 1024 * 256              # launch_argmin's grid cap (1024 CTAs of 256 threads): index LAP + t is thread t again
SMALL_MAX = (4 << 20) // 48   # largest B that cov_argmin evaluates without the sliced pipeline (two UAVs, 48 B a row)


def poll_params(eng, penalty=0.0):
    eng.set_grid_full(16, 16, 1.0, 1.0)
    eng.set_params(2, np.full(2, 3.0), penalty_scale=penalty, prev_xyR=PREV, d_lim=1.0, tan_half_fov=T)


def first_min(obj, feasible, barrier):
    """The documented winner: among the rows the barrier admits, the first index of the smallest objective;
    (+Inf, -1) when the barrier admits none."""
    ok = feasible.astype(bool) if barrier else np.ones(len(obj), dtype=bool)
    if not ok.any():
        return (math.inf, -1)
    m = obj[ok].min()
    return (float(m), int(np.flatnonzero(ok & (obj == m))[0]))


class Multi:
    """cov_multi over two handles on device 0: shard k holds rows [k ceil(B/2), (k+1) ceil(B/2))."""

    def __init__(self, cov):
        self.lib = cov._lib.lib
        self.m = C.c_void_p()
        devs = (C.c_int * 2)(0, 0)
        assert self.lib.cov_multi_create(devs, 2, C.byref(self.m)) == 0

    def params(self, penalty=0.0):
        rm, d_lim = np.full(2, 3.0), np.ones(2)
        for k in range(2):
            h = self.lib.cov_multi_handle(self.m, k)
            assert self.lib.cov_set_grid_full(h, 16, 16, 1.0, 1.0) == 0
            assert self.lib.cov_set_params(h, 2, rm.ctypes.data, penalty, PREV.ctypes.data, d_lim.ctypes.data, T,
                                           0.0, 0) == 0

    def argmin(self, X, barrier):
        X = np.ascontiguousarray(X, dtype=np.float64)
        bo, bi = C.c_double(), C.c_int64()
        assert self.lib.cov_multi_argmin(self.m, X.ctypes.data, len(X), int(barrier), C.byref(bo), C.byref(bi)) == 0
        return (bo.value, bi.value)

    def close(self):
        self.lib.cov_multi_destroy(self.m)


@pytest.fixture()
def poll(cov, engine):
    poll_params(engine)
    multi = Multi(cov)
    multi.params()
    yield engine, multi
    multi.close()


def winners(eng, multi, X, barrier):
    """(objective, index) from every entry point that reduces a poll."""
    out = {"cov_argmin": eng.argmin(X, barrier=barrier),
           "cov_eval_batch_best": eng.eval_batch_best(X, barrier=barrier)["best"],
           "cov_eval_batch_packed": eng.eval_batch_packed(X.astype(np.int16), 1.0, best=True, barrier=barrier)["best"]}
    if multi is not None:
        out["cov_multi_argmin"] = multi.argmin(X, barrier)
    return out


def check_winner(eng, multi, X, barrier, want_idx=None):
    ref = eng.eval_batch(X)
    want = first_min(ref["obj"], ref["feasible"], barrier)
    if want_idx is not None:
        assert want[1] == want_idx, "the set was not built as planned"
    for who, got in winners(eng, multi, X, barrier).items():
        assert got[1] == want[1] and (got[0] == want[0] or (math.isinf(got[0]) and math.isinf(want[0]))), \
            (who, barrier, got, want)


def tie_set(B, lo, hi, barrier, seed):
    """B filler rows; the best row (for this barrier setting) at lo and hi only; decoys that would win if the
    barrier were ignored (barrier on) or that lose (barrier off) before, between and after them."""
    rng = np.random.default_rng(seed)
    X = FILLERS[rng.integers(0, len(FILLERS), B)].copy()
    target, decoy = (BEST_FEASIBLE, BEST_ANY) if barrier else (BEST_ANY, BEST_FEASIBLE)
    for k in (0, lo - 1, (lo + hi) // 2, hi + 1, B - 1):
        if 0 <= k < B and k not in (lo, hi):
            X[k] = decoy
    X[lo] = X[hi] = target
    return X


TIE_PLACEMENTS = [
    # (B, earlier copy, later copy): the later copy must lose every time
    pytest.param(1000, 31, 32, id="lanes-31-32"),
    pytest.param(1000, 255, 256, id="cta-255-256"),
    pytest.param(70 * 256, 1 * 256 + 7, 33 * 256 + 1, id="stage2-same-lane"),
    pytest.param(70 * 256, 34 * 256 + 10, 65 * 256 + 3, id="stage2-across-lanes"),
    pytest.param(1001, 500, 501, id="shard-boundary"),
    pytest.param(SMALL_MAX, 31, SMALL_MAX - 1, id="small-path-last"),
    pytest.param(SMALL_MAX + 1, 31, 32, id="pipelined-path-first"),
    pytest.param(LAP + 100, 5, LAP + 5, id="grid-stride-same-thread"),
    pytest.param(LAP + 100, 7, LAP + 3, id="grid-stride-earlier-in-later-thread"),
    pytest.param(2 * LAP + 9, LAP + 1, LAP + 2, id="grid-stride-second-lap"),
]


@gpu
@pytest.mark.parametrize("barrier", [True, False], ids=["barrier", "no-barrier"])
@pytest.mark.parametrize("B,lo,hi", TIE_PLACEMENTS)
def test_poll_winner_ties(cov, poll, B, lo, hi, barrier):
    eng, multi = poll
    X = tie_set(B, lo, hi, barrier, seed=B + lo)
    check_winner(eng, multi, X, barrier, want_idx=lo)


@gpu
def test_poll_winner_edges(cov, poll):
    eng, multi = poll
    rng = np.random.default_rng(3)
    for B in (1, 33, 1000, LAP + 17):
        same = np.tile(BEST_FEASIBLE, (B, 1))                       # every row identical: index 0
        for barrier in (True, False):
            check_winner(eng, multi, same, barrier, want_idx=0)
        only_last = np.tile(BEST_ANY, (B, 1))                       # only the last row feasible
        only_last[-1] = FILLERS[0]
        check_winner(eng, multi, only_last, True, want_idx=B - 1)
        check_winner(eng, multi, only_last, False, want_idx=0)
        none = np.tile(BEST_ANY, (B, 1))                             # nothing feasible
        none[rng.integers(0, B, max(1, B // 7))] = FILLERS[4]
        check_winner(eng, multi, none, True, want_idx=-1)
        assert eng.argmin(none, barrier=True) == (math.inf, -1)
    # a feasible +Inf objective still wins over the barrier's +Inf: (+Inf, its index), never -1.  With
    # penalty_scale 1e308, |R - r_max| = 1 or 2 on both UAVs gives 2e308 or 4e308 = +Inf through public inputs.
    poll_params(eng, penalty=1e308)
    multi.params(penalty=1e308)
    for B, first in ((1, 0), (40, 17), (LAP + 40, LAP + 11)):
        X = np.tile(BEST_ANY, (B, 1))                                # infeasible, objective +Inf
        X[first:] = np.where(rng.random((B - first, 1)) < 0.5, _row(4, 4), _row(2, 2))  # feasible, +Inf as well
        ref = eng.eval_batch(X)
        assert np.isinf(ref["obj"]).all() and ref["feasible"][first] == 1
        check_winner(eng, multi, X, True, want_idx=first)
        check_winner(eng, multi, X, False, want_idx=0)


@gpu
@pytest.mark.slow
def test_poll_winner_tie_across_host_windows(cov, engine):
    """cov_eval_batch_best / cov_argmin / cov_eval_batch_packed evaluate ~1 GiB of candidates per device window and
    merge the windows' winners on the host.  With 1024 UAVs a window is 2^30 / (24 * 1024) = 43 690 candidates;
    the tie sits on its last row and the next window's first."""
    N = 1024
    window = (1 << 30) // (24 * N)
    B = window + 64
    eng = engine
    pre = np.zeros(3 * N)
    pre[[0, 1]], pre[[N, N + 1]], pre[[2 * N, 2 * N + 1]] = (4.0, 12.0), (8.0, 8.0), (3.0, 3.0)
    eng.set_grid_full(16, 16, 1.0, 1.0)
    eng.set_params(N, np.r_[3.0, 3.0, np.zeros(N - 2)], penalty_scale=0.0, prev_xyR=pre, d_lim=1.0, tan_half_fov=T)
    rng = np.random.default_rng(5)
    Q = np.zeros((B, 3 * N), dtype=np.int16)                       # UAVs 2.. have zero radius: they cover nothing
    Q[:, [0, 1]], Q[:, [N, N + 1]] = (4, 12), (8, 8)
    Q[:, [2 * N, 2 * N + 1]] = FILLERS[rng.integers(0, len(FILLERS), B)][:, 4:6]
    for barrier in (True, False):
        best, decoy = ((4, 4), (5, 5)) if barrier else ((5, 5), (4, 4))
        Qb = Q.copy()
        Qb[[0, window - 2, window + 1], 2 * N:2 * N + 2] = decoy
        Qb[[window - 1, window], 2 * N:2 * N + 2] = best
        r = eng.eval_batch_packed(Qb, 1.0, best=True, barrier=barrier)
        want = first_min(r["obj"], r["feasible"], barrier)
        assert want[1] == window - 1 and r["best"] == want, (barrier, r["best"], want)
        X = Qb.astype(np.float64)
        del Qb
        assert eng.eval_batch_best(X, barrier=barrier)["best"] == want
        assert eng.argmin(X, barrier=barrier) == want
        del X


# ================================================================ 2. fire automaton
EMPTY, TREE, FIRE = 0, 1, 2
SEEDS = [0, 2026, 2 ** 32 + 7, 2 ** 64 - 1]
STEPS = [0, 1, 2 ** 32 - 1, 77]
# cos(1e300 - a) == cos(1e300) for every neighbour angle a (1e300 - a rounds to 1e300), and cos(1e300) < 0:
# wind speed -4 makes every p = -4 cos(1e300) = 2.30 >= 1, so every draw ignites
ALL_IGNITE = (-4.0, 1e300, 1.0)
NONE_IGNITE = (4.0, math.radians(270.0), 0.0)
WINDS = [(4.0, math.radians(a), 0.5) for a in range(0, 360, 45)] + [(3.0, 1.234, 0.37), ALL_IGNITE, NONE_IGNITE]
LATTICES = [(100, 100, 5.0), (37, 91, 5.0), (91, 37, 5.0), (1, 50, 5.0), (2, 50, 5.0), (3, 3, 5.0),
            (600, 700, 1.0)]  # 420 000 cells: more than the 148 * 8 * 256 threads of one grid-stride lap


def cells_of(pts, nx, dx, dy):
    i = np.rint(pts[:, 0] / dx + 0.5).astype(np.int64) - 1
    j = np.rint(pts[:, 1] / dy + 0.5).astype(np.int64) - 1
    return i + nx * j


def histogram(pts, nx, ny, dx, dy):
    h = np.zeros(nx * ny, dtype=np.int64)
    np.add.at(h, cells_of(pts, nx, dx, dy), 1)
    return h


def burning_points(state, nx, dx, dy):
    t = np.flatnonzero(state == FIRE)
    i, j = t % nx + 1, t // nx + 1
    return np.stack([i * dx - dx / 2, j * dy - dy / 2, np.full(len(t), dx * dy), np.full(len(t), dx * dy),
                     np.zeros(len(t))], axis=1)


def random_forest(nx, ny, seed):
    rng = np.random.default_rng(seed)
    s = np.where(rng.random(nx * ny) < 0.7, TREE, EMPTY).astype(np.uint8)
    s[rng.random(nx * ny) < 0.03] = FIRE
    s[0] = FIRE                                             # a corner: on 3 x 3 the one interior cell can still burn
    s[(nx // 2) + nx * (ny // 2)] = TREE
    return s


def check_objective(orc, eng, pts, nx, ny, dx, dy, seed):
    N = 3
    r_max = np.full(N, 30 * T)
    eng.set_params(N, r_max)
    rng = np.random.default_rng(seed)
    X = np.concatenate([rng.random((300, N)) * nx * dx, rng.random((300, N)) * ny * dy,
                        (5 + rng.random((300, N)) * 25) * T * max(dx, dy) / 5], axis=1)
    got = eng.eval_batch(X)
    want = orc.eval_batch(X, N, r_max, pts)
    assert np.array_equal(got["count"], want["count"]) and np.array_equal(got["feasible"], want["feasible"])
    assert np.array_equal(got["obj"].view(np.uint64), want["obj"].view(np.uint64))


@gpu
@pytest.mark.parametrize("push_initial", [1, 0])
@pytest.mark.parametrize("nx,ny,d", LATTICES, ids=[f"{a}x{b}" for a, b, _ in LATTICES])
def test_fire_automaton_lattices(cov, orc, engine, nx, ny, d, push_initial):
    """Every step: the state, the number of pushed entries and the store's multiplicities equal the C oracle's.
    Seeds, step counters, winds and the append flag rotate through their edge values."""
    state = random_forest(nx, ny, seed=nx * 1000 + ny)
    engine.fire_init(state, nx, ny, d, d, push_initial=bool(push_initial))
    pts = burning_points(state, nx, d, d) if push_initial else np.zeros((0, 5))
    mult = histogram(pts, nx, ny, d, d)
    assert np.array_equal(engine.grid_cells(), mult)
    grid = state.copy()
    total = 0
    for k in range(len(WINDS) + 1):
        seed, step = SEEDS[k % 4], STEPS[(k + k // 4) % 4]
        ws, wd, ps = WINDS[k % len(WINDS)]
        append = k % 3 != 2
        pushed = engine.fire_step(ws, wd, ps, seed=seed, step=step, append=append)
        grid, new = orc.fire_step(grid, nx, ny, d, d, ws, wd, ps, step, seed)
        assert pushed == len(new), (k, pushed, len(new))
        assert np.array_equal(engine.fire_state(), grid), k
        if append:
            pts = np.concatenate([pts, new])
            mult += histogram(new, nx, ny, d, d)
        assert np.array_equal(engine.grid_cells(), mult), k
        assert engine.grid_info()["n_entries"] == len(pts)
        if (ws, wd, ps) == NONE_IGNITE:
            assert pushed == 0
        total += pushed
    if nx >= 3 and ny >= 3:
        assert total > 0
    else:
        assert total == 0 and np.array_equal(grid, state)  # no interior cell
    check_objective(orc, engine, pts, nx, ny, d, d, seed=nx + ny)
    with pytest.raises(cov.CoverageError) as ei:
        engine.fire_step(4.0, 0.0, 0.5, seed=1, step=2 ** 32)
    assert ei.value.code == cov._lib.COV_ERR_INVALID
    with pytest.raises(cov.CoverageError) as ei:
        engine.fire_step(4.0, 0.0, 0.5, seed=1, step=-1)
    assert ei.value.code == cov._lib.COV_ERR_INVALID
    assert np.array_equal(engine.fire_state(), grid)


@gpu
def test_fire_overflow_leaves_everything_as_it_was(cov, orc, engine):
    """A step that would put a 256th entry on a cell returns COV_ERR_LIMIT and changes nothing; once the cell is
    emptied, the same step runs and matches the oracle."""
    nx, ny, d = 37, 23, 5.0
    state = np.full(nx * ny, TREE, dtype=np.uint8)
    fire = 10 + nx * 7
    target = fire + 1                                   # the TREE cell next to the burning one
    state[fire] = FIRE
    state[5 + nx * 15] = FIRE
    engine.fire_init(state, nx, ny, d, d, push_initial=True)
    full = np.repeat(burning_points(np.where(np.arange(nx * ny) == target, FIRE, EMPTY), nx, d, d), 255, axis=0)
    engine.add_points(full)
    pts = np.concatenate([burning_points(state, nx, d, d), full])
    N = 3
    engine.set_params(N, np.full(N, 30 * T))
    rng = np.random.default_rng(1)
    X = np.concatenate([rng.random((200, 2 * N)) * 150, (5 + rng.random((200, N)) * 25) * T], axis=1)
    before = (engine.fire_state(), engine.grid_cells(), engine.grid_info(), engine.eval_batch(X))
    assert before[1][target] == 255
    ws, wd, ps = ALL_IGNITE
    with pytest.raises(cov.CoverageError) as ei:
        engine.fire_step(ws, wd, ps, seed=2 ** 40 + 3, step=9)
    assert ei.value.code == cov._lib.COV_ERR_LIMIT
    after = (engine.fire_state(), engine.grid_cells(), engine.grid_info(), engine.eval_batch(X))
    assert np.array_equal(after[0], before[0]) and np.array_equal(after[1], before[1]) and after[2] == before[2]
    for k in ("obj", "count", "feasible"):
        assert np.array_equal(after[3][k], before[3][k]), k
    tx, ty = (target % nx + 1) * d - d / 2, (target // nx + 1) * d - d / 2
    assert engine.remove_covered([tx, ty, 1.0]) == 255
    pts = pts[cells_of(pts, nx, d, d) != target]
    pushed = engine.fire_step(ws, wd, ps, seed=2 ** 40 + 3, step=9)
    grid, new = orc.fire_step(state, nx, ny, d, d, ws, wd, ps, 9, 2 ** 40 + 3)
    assert pushed == len(new) > 0 and np.array_equal(engine.fire_state(), grid)
    pts = np.concatenate([pts, new])
    assert np.array_equal(engine.grid_cells(), histogram(pts, nx, ny, d, d))
    check_objective(orc, engine, pts, nx, ny, d, d, seed=4)


def update_grid_numpy(synth, grid, nx, ny, dx, dy, wind_speed, wind_direction, prob_spread, step, seed):
    """src/DynamicArea.jl:52-72 transcribed: `for i in 2:nx-1, j in 2:ny-1` (j fastest); an interior TREE cell
    draws once per burning neighbour of its 3x3 window, in findall's column-major order (a fastest), and every
    success sets FIRE and pushes [i dx - dx/2, j dy - dy/2, dx dy, dx dy, false].  rand() is the Philox4x32-10
    uniform of counter (cell low, step, (a-1) + 3(b-1), cell high) and key (seed low, seed high), synth._philox."""
    g = np.asarray(grid, dtype=np.uint8).reshape(ny, nx).T      # g[i-1, j-1]
    new = g.copy()
    pts = []
    for i in range(2, nx):
        for j in range(2, ny):
            if g[i - 1, j - 1] != TREE:
                continue
            for b in range(1, 4):
                for a in range(1, 4):
                    if g[i - 2 + a - 1, j - 2 + b - 1] != FIRE:
                        continue
                    p = wind_speed * math.cos(wind_direction - math.atan2(2 - b, 2 - a)) * prob_spread
                    cell = (i - 1) + nx * (j - 1)
                    r = synth._philox(cell & 0xFFFFFFFF, step, (a - 1) + 3 * (b - 1), cell >> 32,
                                      seed & 0xFFFFFFFF, seed >> 32)
                    u = float(synth._u01_53(r[0], r[1]))
                    if p > u:
                        new[i - 1, j - 1] = FIRE
                        pts.append([i * dx - dx / 2, j * dy - dy / 2, dx * dy, dx * dy, 0.0])
    return new.T.ravel(), np.array(pts, dtype=np.float64).reshape(-1, 5)


def test_fire_oracle_matches_numpy_transcription(cov, orc):
    """The C oracle the device is checked against is itself right off the diagonal: a non-square lattice (a swap
    of i/j or nx/ny shows) and seeds with a non-zero high word."""
    nx, ny, d = 23, 41, 5.0
    grid = random_forest(nx, ny, seed=8)
    for seed, step, wind in ((2 ** 64 - 1, 2 ** 32 - 1, (4.0, math.radians(300.0), 0.5)),
                             (2 ** 32 + 7, 0, (3.0, 1.234, 0.37)), (11, 5, ALL_IGNITE)):
        want_grid, want_pts = update_grid_numpy(cov.synth, grid, nx, ny, d, d, *wind, step, seed)
        got_grid, got_pts = orc.fire_step(grid, nx, ny, d, d, *wind, step, seed)
        assert np.array_equal(got_grid, want_grid) and np.array_equal(got_pts, want_pts)
        assert len(want_pts) > 0
        grid = want_grid


# ================================================================ 3. cell removal and covered mask
def createpoi_cell_index(nx, ny):
    """Cell (i-1) + nx (j-1) of every entry of createPOI(dx, dy, nx, ny): i outer, j inner."""
    return (np.arange(nx)[:, None] + nx * np.arange(ny)[None, :]).ravel()


def reference_mask(npo, x, nx, ny, dx, dy):
    """coverage_oracle.covered_mask (the reference predicate sqrt(s) < R) on the full createPOI list, per cell."""
    mask = np.zeros(nx * ny, dtype=np.uint8)
    mask[createpoi_cell_index(nx, ny)] = npo.covered_mask(np.asarray(x, dtype=np.float64), npo.createPOI(dx, dy, nx, ny))
    return mask


def centre_on_threshold(orc, px, py, R, where):
    """A disc centre whose radicand fl(fl((px-cx)^2) + fl((py-cy)^2)) at the cell centre (px, py) is T(R) one ulp
    down (where = -1: covered), T(R) itself (0: not covered, the predicate is strict) or one ulp up (+1).  The
    centre sits left of the cell, with fl((px-cx)^2) just below the target; a tiny ddy = n ulp(py) supplies the
    rest, in steps far finer than an ulp of the radicand."""
    t = orc.threshold_by_search(R)
    want = {-1: math.nextafter(t, -math.inf), 0: t, 1: math.nextafter(t, math.inf)}[where]
    cx = px - math.sqrt(want)
    while (px - cx) * (px - cx) >= want:
        cx = math.nextafter(cx, math.inf)
    a = (px - cx) * (px - cx)
    u = math.ulp(py)
    n0 = round(math.sqrt(want - a) / u)
    for n in sorted(range(max(0, n0 - 500), n0 + 501), key=lambda n: abs(n - n0)):
        cy = py - n * u
        if a + (py - cy) * (py - cy) == want:
            return cx, cy
    raise AssertionError(f"no centre puts the radicand on T({R!r}) {where:+d} ulp")


BOUNDARY_RADII = (7.3, 8.0, 12.345678901234567, 2.5)   # 8.0: a power of two, the closed form's other branch


def boundary_discs(orc, nx, ny, dx, dy, seed):
    """Discs that each put one cell's radicand exactly on T(R) or one ulp either side; returns (x, [(cell, covered)])."""
    rng = np.random.default_rng(seed)
    xs, ys, rs, probes = [], [], [], []
    for R in BOUNDARY_RADII:
        for where in (-1, 0, 1):
            i = int(rng.integers(max(1, nx // 4), max(2, 3 * nx // 4))) + 1
            j = int(rng.integers(max(1, ny // 4), max(2, 3 * ny // 4))) + 1
            px, py = i * dx - dx / 2, j * dy - dy / 2
            cx, cy = centre_on_threshold(orc, px, py, R, where)
            xs.append(cx)
            ys.append(cy)
            rs.append(R)
            probes.append(((i - 1) + nx * (j - 1), where < 0))
    return np.array(xs + ys + rs), probes


def disc_sets(orc, nx, ny, dx, dy, seed):
    """The disc sets every removal / mask test runs: (name, [x; y; R])."""
    rng = np.random.default_rng(seed)
    lx, ly = nx * dx, ny * dy
    ext = 0.15 * max(lx, ly)

    def rand(N, rmin, rmax):
        return np.concatenate([rng.random(N) * lx, rng.random(N) * ly, rmin + rng.random(N) * (rmax - rmin)])

    sets = [("boundary", boundary_discs(orc, nx, ny, dx, dy, seed)[0])]
    z = rand(6, 0.5 * ext, ext)
    z[12:15] = 0.0                                          # three of six discs with R = 0
    sets.append(("zero-radius", z))
    off = np.array([-10 * lx, 3 * lx, lx / 2, -ext - 1, ly / 2, 5 * ly, ext, ext, 2 * ext])  # wholly off the grid
    sets.append(("off-grid", off))
    sets.append(("N=1", rand(1, ext, 2 * ext)))
    sets.append(("N=33", rand(33, 0.1 * ext, 0.6 * ext)))
    sets.append(("N=1024", rand(1024, 0.0, 0.05 * ext)))
    return sets


MASK_LATTICES = [(37, 91, 5.0, 5.0), (91, 37, 5.0, 2.5), (600, 700, 1.0, 1.0)]


def test_threshold_matches_definition(cov, orc):
    for R in BOUNDARY_RADII + (0.0, 1e-3, 1e3, 31.0 * T, 2.0 ** -30, 2.0 ** 20 + 1):
        assert cov.engine.threshold(R) == orc.threshold_by_search(R), R


def test_boundary_discs_straddle_the_threshold(orc, npo):
    """The boundary set is what it claims: at every probe cell the reference predicate flips exactly there."""
    nx, ny, d = 37, 91, 5.0
    x, probes = boundary_discs(orc, nx, ny, d, d, seed=1)
    n = len(x) // 3
    for k, (cell, covered) in enumerate(probes):
        i, j = cell % nx + 1, cell // nx + 1
        px, py = i * d - d / 2, j * d - d / 2
        s = (px - x[k]) * (px - x[k]) + (py - x[n + k]) * (py - x[n + k])
        t = orc.threshold_by_search(x[2 * n + k])
        assert s in (np.nextafter(t, -np.inf), t, np.nextafter(t, np.inf))
        assert bool(math.sqrt(s) < x[2 * n + k]) == covered == (s < t)


@gpu
@pytest.mark.parametrize("nx,ny,dx,dy", MASK_LATTICES, ids=[f"{a}x{b}" for a, b, _, _ in MASK_LATTICES])
def test_covered_mask_cell_by_cell(cov, orc, npo, engine, nx, ny, dx, dy):
    engine.set_grid_full(nx, ny, dx, dy)
    for name, x in disc_sets(orc, nx, ny, dx, dy, seed=nx):
        N = len(x) // 3
        if nx * ny > 100_000 and N > 64:
            continue                                        # (the NumPy predicate over 420 000 cells x 1024 discs)
        engine.set_params(N, np.zeros(N))
        got = engine.covered_mask(x)
        want = reference_mask(npo, x, nx, ny, dx, dy)
        assert np.array_equal(got, want), (name, np.flatnonzero(got != want)[:10])
        if name == "boundary":                              # each disc alone: its probe cell flips exactly at T(R)
            engine.set_params(1, np.zeros(1))
            for k, (cell, covered) in enumerate(boundary_discs(orc, nx, ny, dx, dy, seed=nx)[1]):
                one = x[k::N]
                got1 = engine.covered_mask(one)
                assert got1[cell] == covered, (k, one)
                assert np.array_equal(got1, reference_mask(npo, one, nx, ny, dx, dy)), k
        if name == "off-grid":
            assert not got.any()


def store_stats(pts, nx, ny, dx, dy, cls_of_weight):
    """(multiplicities, n_planes) of a list: planes = the set bits of the OR of each class's multiplicities."""
    mult = histogram(pts, nx, ny, dx, dy)
    planes = 0
    for w in cls_of_weight:
        m = np.zeros(nx * ny, dtype=np.int64)
        sel = pts[:, 3] == w
        np.add.at(m, cells_of(pts[sel], nx, dx, dy), 1)
        planes += bin(int(np.bitwise_or.reduce(m))).count("1")
    return mult, max(planes, 1)


def list_with_multiplicities(nx, ny, dx, dy, seed, classes):
    """A shuffled list: `classes` = [(weight, allowed multiplicities)], each on its own random cells."""
    rng = np.random.default_rng(seed)
    cells = rng.permutation(nx * ny)
    rows, at = [], 0
    for w, mults in classes:
        take = cells[at:at + nx * ny // (2 * len(classes))]
        at += len(take)
        m = rng.choice(np.asarray(mults), len(take))
        m[:len(mults)] = mults                              # every allowed multiplicity occurs
        c = np.repeat(take, m)
        i, j = c % nx + 1, c // nx + 1
        rows.append(np.stack([i * dx - dx / 2, j * dy - dy / 2, np.full(len(c), dx * dy), np.full(len(c), w),
                              np.zeros(len(c))], axis=1))
    pts = np.concatenate(rows)
    return pts[rng.permutation(len(pts))]


@gpu
@pytest.mark.parametrize("store", ["points-two-classes", "points-255", "grid-bits-big"])
def test_remove_covered_matches_rmvCoveredPOI(cov, orc, engine, store):
    """After every removal: the count removed, the multiplicities and the grid info equal rmvCoveredPOI on the list;
    at the end the objective equals the oracle's on the surviving list."""
    if store == "points-two-classes":
        nx, ny, dx, dy = 37, 91, 5.0, 5.0
        classes = [(25.0, list(range(16, 256, 16))), (6.25, list(range(1, 16)))]   # 4 + 4 bit planes
        pts = list_with_multiplicities(nx, ny, dx, dy, 7, classes)
        engine.set_points(pts, nx, ny, dx, dy)
    elif store == "points-255":
        nx, ny, dx, dy = 91, 37, 5.0, 5.0
        classes = [(25.0, [255, 254, 253, 128, 127, 1, 2, 200])]
        pts = list_with_multiplicities(nx, ny, dx, dy, 8, classes)
        engine.set_points(pts, nx, ny, dx, dy)
    else:
        nx, ny, dx, dy = 600, 700, 1.0, 1.0                 # 420 000 cells: more than one grid-stride lap
        rng = np.random.default_rng(9)
        fire = rng.random((nx, ny)) < 0.5
        bits = cov.synth.pack_bits(fire)
        pts = cov.synth.points_from_bits(bits, nx, dx, dy)
        classes = [(1.0, [1])]
        engine.set_grid_bits(bits, nx, ny, dx, dy)
    weights = [w for w, _ in classes]
    info0 = engine.grid_info()
    assert info0["n_entries"] == len(pts) and info0["n_classes"] == len(classes)
    for name, x in disc_sets(orc, nx, ny, dx, dy, seed=nx * 3 + ny):
        keep = orc.rmvCoveredPOI(x, pts)
        removed = engine.remove_covered(x)
        assert removed == len(pts) - len(keep), name
        pts = keep
        mult, planes = store_stats(pts, nx, ny, dx, dy, weights)
        assert np.array_equal(engine.grid_cells(), mult), name
        info = engine.grid_info()
        assert (info["n_entries"], info["n_cells"], info["n_planes"], info["n_classes"]) == \
            (len(pts), int((mult > 0).sum()), planes, len(classes)), (name, info)
        assert (info["nx"], info["ny"], info["dx"], info["dy"], info["area_exact"]) == \
            (nx, ny, dx, dy, info0["area_exact"])
    assert 0 < len(pts) < info0["n_entries"]
    check_objective(orc, engine, pts, nx, ny, dx, dy, seed=3)


# ================================================================ 4. union area
def _dedup(x):
    """Discs with R > 0, exact duplicates dropped (the union does not change)."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x) // 3
    seen, out = set(), []
    for i in range(n):
        d = (float(x[i]), float(x[n + i]), float(x[2 * n + i]))
        if d[2] > 0 and d not in seen:
            seen.add(d)
            out.append(d)
    return out


def union_area_mp(x, dps=60):
    """Area of the union of the discs [x; y; R] in mpmath, by point tests: every circle is cut at every angle where
    it meets another circle (tangent points included), and an arc between two cuts is exposed iff its MIDPOINT lies
    strictly inside no other disc.  The exposed arcs are summed with Green's formula
    1/2 [R^2 (t2 - t1) + R (cx (sin t2 - sin t1) - cy (cos t2 - cos t1))].  The doubles are exact in mpmath, so
    tangency and containment are decided exactly; no interval merging and no tie rule is involved."""
    import mpmath as mp
    discs = _dedup(x)
    with mp.workdps(dps):
        two_pi = 2 * mp.pi
        M = [(mp.mpf(a), mp.mpf(b), mp.mpf(r)) for a, b, r in discs]
        total = mp.mpf(0)
        for i, (xi, yi, ri) in enumerate(M):
            fi = discs[i]
            cuts, near = [mp.mpf(0)], []
            for j, (xj, yj, rj) in enumerate(M):
                fj = discs[j]
                if j == i or math.hypot(fj[0] - fi[0], fj[1] - fi[1]) > (fi[2] + fj[2]) * (1 + 1e-9):
                    continue                                # far apart (decided exactly below when close)
                dx, dy = xj - xi, yj - yi
                d2 = dx * dx + dy * dy
                if d2 >= (ri + rj) ** 2:
                    continue                                # apart or externally tangent: no point strictly inside
                near.append((xj, yj, rj))
                if d2 == 0:
                    continue
                d = mp.sqrt(d2)
                c = (ri * ri + d2 - rj * rj) / (2 * ri * d)
                if abs(c) <= 1:
                    phi, al = mp.atan2(dy, dx), mp.acos(c)
                    cuts += [(phi - al) % two_pi, (phi + al) % two_pi]
            cuts = sorted(set(cuts)) + [two_pi]
            for t1, t2 in zip(cuts, cuts[1:]):
                tm = (t1 + t2) / 2
                px, py = xi + ri * mp.cos(tm), yi + ri * mp.sin(tm)
                if any((px - xj) ** 2 + (py - yj) ** 2 < rj * rj for xj, yj, rj in near):
                    continue
                total += (ri * ri * (t2 - t1) + ri * (xi * (mp.sin(t2) - mp.sin(t1)) - yi * (mp.cos(t2) - mp.cos(t1)))) / 2
        return float(total)


UNION_K = 64  # rounding errors per Green term (a dozen operations, two sincos, the sum over arcs and circles)


def union_error_bound(x):
    """What an FP64 boundary integration may be off by, derived from its operations.  Per circle i, the Green terms
    are of size s_i = R_i (R_i + |cx_i| + |cy_i|) / 2 per radian, and |d term / d endpoint| <= s_i.  Two sources:
      - rounding in the terms and their sums: UNION_K eps s_i (2 pi + 2 m_i), m_i = circles that meet circle i;
      - the angle of every cut: atan2 and fmod (8 eps), and acos of c = (Ri^2 + d^2 - Rj^2) / (2 Ri d), whose
        rounding error is at most dc = 16 eps (Ri^2 + d^2 + Rj^2) / (2 Ri d).  acos turns dc into at most
        min(dc / sqrt(1 - (|c| + dc)^2), pi/2 sqrt(dc)): a multiple of eps for well-separated cuts, sqrt(eps) near
        tangency, where a cut moves along the circle by that much whichever way the containment tests go.
    Returns the bound sum_i [UNION_K eps s_i (2 pi + 2 m_i) + sum_j 2 s_i (dalpha_ij + 8 eps)]."""
    discs = _dedup(x)
    bound = 0.0
    for i, (xi, yi, ri) in enumerate(discs):
        s = 0.5 * ri * (ri + abs(xi) + abs(yi))
        m = 0
        for j, (xj, yj, rj) in enumerate(discs):
            if j == i:
                continue
            d = math.hypot(xj - xi, yj - yi)
            if d > (ri + rj) * (1 + 1e-12) or d == 0.0:
                continue
            m += 1
            dc = 16 * EPS * (ri * ri + d * d + rj * rj) / (2 * ri * d)
            c = (ri * ri + d * d - rj * rj) / (2 * ri * d)
            if abs(c) > 1 + dc:
                continue                                     # nested without touching: no cut
            room = 1 - (abs(c) + dc) ** 2
            da = 0.5 * math.pi * math.sqrt(dc)
            if room > 0:
                da = min(da, dc / math.sqrt(room))
            bound += 2 * s * (da + 8 * EPS)
        bound += UNION_K * EPS * s * (2 * math.pi + 2 * m)
    return bound


def lens_union(r1, r2, d):
    """Closed form: the union of two discs of radii r1, r2 whose centres are d apart."""
    if d >= r1 + r2:
        return math.pi * (r1 * r1 + r2 * r2)
    if d <= abs(r1 - r2):
        return math.pi * max(r1, r2) ** 2
    a1 = math.acos((d * d + r1 * r1 - r2 * r2) / (2 * d * r1))
    a2 = math.acos((d * d + r2 * r2 - r1 * r1) / (2 * d * r2))
    k = 0.5 * math.sqrt((-d + r1 + r2) * (d + r1 - r2) * (d - r1 + r2) * (d + r1 + r2))
    return math.pi * (r1 * r1 + r2 * r2) - (r1 * r1 * a1 + r2 * r2 * a2 - k)


def discs(*circles):
    """[(x, y, R), ...] -> [x; y; R]."""
    c = np.array(circles, dtype=np.float64).reshape(-1, 3)
    return np.concatenate([c[:, 0], c[:, 1], c[:, 2]])


def slab_area(x):
    """Area of the union by integrating, over x, the length of the union of the discs' vertical chords (mpmath
    tanh-sinh quadrature between the abscissae where that union changes shape)."""
    import mpmath as mp
    ds = _dedup(x)
    with mp.workdps(30):
        D = [(mp.mpf(a), mp.mpf(b), mp.mpf(r)) for a, b, r in ds]
        xs = set()
        for a, b, r in D:
            xs |= {a - r, a + r}
        for i, (a, b, r) in enumerate(D):                  # abscissae of the intersection points
            for (a2, b2, r2) in D[i + 1:]:
                dx, dy = a2 - a, b2 - b
                d = mp.sqrt(dx * dx + dy * dy)
                if 0 < d < r + r2 and d > abs(r - r2):
                    l = (r * r - r2 * r2 + d * d) / (2 * d)
                    h = mp.sqrt(max(r * r - l * l, 0))
                    xs |= {a + l * dx / d - h * dy / d, a + l * dx / d + h * dy / d}
        xs = sorted(xs)

        def length(t):
            iv = sorted((b - mp.sqrt(r * r - (t - a) ** 2), b + mp.sqrt(r * r - (t - a) ** 2))
                        for a, b, r in D if abs(t - a) < r)
            tot, lo, hi = mp.mpf(0), None, None
            for p, q in iv:
                if hi is None or p > hi:
                    if hi is not None:
                        tot += hi - lo
                    lo, hi = p, q
                else:
                    hi = max(hi, q)
            return tot + (hi - lo if hi is not None else 0)

        return float(sum(mp.quad(length, [p, q]) for p, q in zip(xs, xs[1:])))


def union_edge_cases():
    """(name, [x; y; R]) at the edges of the boundary integration."""
    cases = []
    for r1, r2 in ((1.0, 1.0), (1.5, 0.7), (3.0, 1e-3)):
        for th in (0.0, 0.7, math.pi / 2):
            ux, uy = math.cos(th), math.sin(th)
            for base, kind in ((r1 + r2, "external"), (abs(r1 - r2), "internal")):
                if base == 0.0:
                    continue
                for k in range(-4, 5):
                    d = base
                    for _ in range(abs(k)):
                        d = math.nextafter(d, math.inf if k > 0 else -math.inf)
                    cases.append((f"{kind}-tangent{k:+d}ulp-{r1}-{r2}-{th:.2f}", discs((0.3, -0.2, r1),
                                                                                  (0.3 + d * ux, -0.2 + d * uy, r2))))
    r = 2.0                                                 # three circles through the origin
    cases.append(("common-point", discs(*[(r * math.cos(a), r * math.sin(a), r) for a in (0.1, 2.2, 4.3)])))
    cases.append(("covered-by-three-not-one", discs((0, 0, 1.0), *[(1.2 * math.cos(a), 1.2 * math.sin(a), 1.0)
                                                                  for a in (0.0, 2 * math.pi / 3, 4 * math.pi / 3)])))
    cases.append(("two-identical-cut-a-third", discs((0, 0, 1.0), (1.2, 0.3, 0.8), (1.2, 0.3, 0.8))))
    cases.append(("three-identical-cut-two", discs((1.2, 0.3, 0.8), (0, 0, 1.0), (1.2, 0.3, 0.8), (0.5, 1.5, 1.1),
                                                   (1.2, 0.3, 0.8))))
    cases.append(("identical-pairs-shared-ends", discs((0, 0, 1.0), (1.0, 0, 1.0), (1.0, 0, 1.0), (0, 1.0, 1.0),
                                                       (0, 1.0, 1.0), (0, 0, 1.0))))
    cases.append(("concentric-stack", discs(*[(2.0, 3.0, float(k)) for k in range(1, 9)])))
    cases.append(("concentric-stack-cut", discs(*[(2.0, 3.0, float(k)) for k in (1, 2, 3)], (5.5, 3.0, 1.0))))
    cases.append(("wrap-right", discs((0, 0, 1.0), (1.5, 0.0, 1.0))))           # an interval across angle 0
    cases.append(("wrap-right-below", discs((0, 0, 1.0), (1.2, -1e-9, 0.5))))
    cases.append(("wrap-left", discs((0, 0, 1.0), (-1.5, 0.0, 1.0))))
    cases.append(("wrap-both", discs((0, 0, 1.0), (1.5, 0.0, 1.0), (0.9, 0.9, 0.6), (1.1, -0.7, 0.6))))
    big = [(0.0, 0.0, 1e3)]                                 # tiny discs on, just inside and just outside a huge one
    for k, a in enumerate(np.linspace(0, 2 * math.pi, 7)[:-1]):
        rr = 1e3 + (0.0, 5e-7, -5e-7, 2e-6, 1e-7, -2e-6)[k]
        big.append((rr * math.cos(a), rr * math.sin(a), 1e-6))
    cases.append(("tiny-next-to-huge", discs(*big)))
    cases.append(("tiny-next-to-huge-offset", discs((1e3, -2e3, 1e3), (1e3 + 1e3, -2e3, 1e-6), (1e3, -1e3 + 1e-6, 1e-6))))
    return cases


def random_swarm(rng, N, spread=None):
    spread = spread if spread is not None else 8.0 * math.sqrt(N)
    return np.concatenate([rng.random(2 * N) * spread, 1.0 + rng.random(N) * 4.0])


def pad(x, n_to):
    n = len(x) // 3
    z = np.zeros(n_to - n)
    return np.concatenate([x[:n], z, x[n:2 * n], z, x[2 * n:], z])


def test_union_reference_closed_forms():
    lens = lambda d: lens_union(1.0, 1.0, d)  # noqa: E731
    for x, want in [(discs((0, 0, 1.0)), math.pi), (discs((0, 0, 1.0), (1.0, 0, 1.0)), lens(1.0)),
                    (discs((0, 0, 1.0), (0.1, 0, 2.0)), 4 * math.pi), (discs((0, 0, 1.0), (0, 0, 1.0)), math.pi),
                    (discs((0, 0, 1.0), (2.0, 0, 1.0)), 2 * math.pi), (discs((0, 0, 1.0), (1.0, 0, 2.0)), 4 * math.pi),
                    (discs((0, 0, 2.0), (5.0, 0, 1.0)), 5 * math.pi), (discs((0, 0, 1.0), (1.0, 0, 0.0)), math.pi),
                    (discs((3, 7, 2.0), (3, 7, 2.0), (3, 7, 2.0)), 4 * math.pi),
                    (discs((0.3, 0.1, 1.7), (1.9, -0.4, 0.6)), lens_union(1.7, 0.6, math.hypot(1.6, 0.5))),
                    (discs(*[(2.0, 3.0, float(k)) for k in range(1, 9)]), 64 * math.pi)]:
        assert abs(union_area_mp(x) - want) <= 1e-14 * want, (x, union_area_mp(x), want)


@pytest.mark.parametrize("N", [2, 3, 4])
def test_union_reference_against_slab_integration(N):
    rng = np.random.default_rng(N)
    for k in range(3):
        x = random_swarm(rng, N, spread=4.0)
        a, b = union_area_mp(x), slab_area(x)
        assert abs(a - b) <= 1e-12 * a, (x, a, b)
    for name, x in union_edge_cases():
        if len(x) // 3 <= 4 and name.startswith(("common", "two-identical", "wrap", "concentric-stack-cut")):
            a, b = union_area_mp(x), slab_area(x)
            assert abs(a - b) <= 1e-12 * a, (name, a, b)


def test_union_bound_covers_the_numpy_restatement(npo):
    """The FP64 NumPy restatement (the kernels' arithmetic with the host's libm) stays inside union_error_bound of
    the mpmath reference on every edge case and on random swarms -- the bound is neither too tight nor vacuous."""
    worst = 0.0
    rng = np.random.default_rng(11)
    cases = union_edge_cases() + [(f"rand{N}", random_swarm(rng, N)) for N in (5, 20, 33) for _ in range(2)]
    for name, x in cases:
        ref, got, bound = union_area_mp(x), npo.union_area(x), union_error_bound(x)
        assert abs(got - ref) <= bound, (name, got, ref, bound)
        assert bound <= 1e-6 * ref, (name, bound, ref)
        worst = max(worst, abs(got - ref) / bound)
    assert worst > 0.0


def union_both_kernels(engine, x, n_big=70):
    """Area of one candidate through the warp kernel (N <= 64) and the CTA kernel (padded with zero-radius discs)."""
    n = len(x) // 3
    out = []
    if n <= 64:
        out.append(("warp", float(engine.union_area(x[None, :], n)[0])))
    nb = max(n_big, n)
    out.append(("cta", float(engine.union_area(pad(x, nb)[None, :], nb)[0])))
    return out


@gpu
def test_union_area_edges_against_mpmath(engine):
    worst = 0.0
    for name, x in union_edge_cases():
        ref, bound = union_area_mp(x), union_error_bound(x)
        for kernel, got in union_both_kernels(engine, x):
            assert abs(got - ref) <= bound, (name, kernel, got, ref, bound)
            worst = max(worst, abs(got - ref) / bound)
    print(f"union area edge cases: worst |kernel - mpmath| / bound = {worst:.3g}")


@gpu
@pytest.mark.parametrize("N", [1, 31, 32, 33, 63, 64, 65, 96, 1024])
def test_union_area_swarm_sizes(npo, engine, N):
    rng = np.random.default_rng(N)
    X = np.stack([random_swarm(rng, N), random_swarm(rng, N, spread=2.0 * math.sqrt(N)),
                  random_swarm(rng, N, spread=30.0 * math.sqrt(N))])
    got = engine.union_area(X, N)
    for b, x in enumerate(X):
        bound = union_error_bound(x)
        ref = union_area_mp(x) if N <= 128 else npo.union_area(x)
        slack = 1 if N <= 128 else 2                      # (the NumPy restatement carries its own rounding)
        assert abs(got[b] - ref) <= slack * bound, (N, b, got[b], ref, bound)
    if N <= 64:
        got_big = engine.union_area(np.stack([pad(x, 70) for x in X]), 70)
        for b, x in enumerate(X):
            assert abs(got_big[b] - got[b]) <= 2 * union_error_bound(x), (N, b)


@gpu
@pytest.mark.parametrize("N,B", [(2, 9472 * 2 + 37), (65, 592 * 2 + 5)], ids=["warp-kernel", "cta-kernel"])
def test_union_area_grid_stride_laps(engine, N, B):
    """More candidates than one launch has warps (9472) or CTAs (592): every row is a different pair of discs
    whose union has a closed form, so a row a lap missed or a row read from the wrong place shows."""
    rng = np.random.default_rng(B)
    r1 = 1.0 + rng.random(B) * 3.0
    r2 = 0.5 + rng.random(B) * 2.0
    d = rng.random(B) * (r1 + r2 + 2.0)
    th = rng.random(B) * 2 * math.pi
    cx, cy = rng.random(B) * 20 - 10, rng.random(B) * 20 - 10
    X = np.zeros((B, 3 * N))
    X[:, 0], X[:, N], X[:, 2 * N] = cx, cy, r1
    X[:, 1], X[:, N + 1], X[:, 2 * N + 1] = cx + d * np.cos(th), cy + d * np.sin(th), r2
    got = engine.union_area(X, N)
    for b in range(B):
        x = np.array([X[b, 0], X[b, 1], X[b, N], X[b, N + 1], X[b, 2 * N], X[b, 2 * N + 1]])
        want = lens_union(r1[b], r2[b], math.hypot(x[1] - x[0], x[3] - x[2]))
        assert abs(got[b] - want) <= union_error_bound(x) + 1e-13 * want, (b, got[b], want)
