"""The list-order area over every way a cell store is built and changed.

With a non-dyadic weight in the store (the high-interest weight (h_max tan(FOV/2))^2 pi, src/CellFunctions.jl:41-45)
the reference's Float64 area depends on the order in which its `points_of_interest` loop adds the weights, and the
library replays that order with the ordered kernel.  `RefList` below is the reference's list as the reference
changes it (createPOI, update_POI's push!, rmvCoveredPOI, the fire automaton); after every operation on a device
store, the store's statistics and every output of the evaluation must equal the C oracle run on that list, bit for
bit.  The CPU part checks the model itself against the oracle."""
import ctypes as C
import math

import numpy as np
import pytest

T = math.tan((100 / 180 * math.pi) / 2)
NX = NY = 40
DX = DY = 5.0
W = DX * DY                              # createPOI / fire weight (dyadic)
H = (30.0 * T) ** 2 * math.pi            # high-interest weight (not dyadic)
H2 = (20.0 * T) ** 2 * math.pi           # a second non-dyadic weight
N = 4
R_MAX = np.full(N, 36.0)
ORDERED = 5
WIND = (4.0, math.radians(270.0), 0.5)


# ---------------------------------------------------------------- the reference's list
def createpoi_cells(nx, ny):
    """Flat cell indices (i-1) + nx*(j-1) in createPOI's order: i outer, j inner (src/AreaCoverageCalculation.jl:14-15)."""
    return (np.arange(nx)[:, None] + nx * np.arange(ny)[None, :]).ravel()


def rows(cells, w, nx=NX, dx=DX, dy=DY):
    cells = np.asarray(cells, dtype=np.int64)
    i, j = cells % nx + 1, cells // nx + 1
    return np.stack([i * dx - dx / 2, j * dy - dy / 2, np.full(len(cells), dx * dy),
                     np.full(len(cells), float(w)), np.zeros(len(cells))], axis=1)


def area_exact_rule(weights, n_entries):
    """cov_grid_info.area_exact restated: every weight's odd mantissa, scaled to the smallest exponent, times
    n_entries, summed over the classes, stays below 2^53; weight 0 is skipped; a negative, +Inf or NaN weight fails."""
    parts = []
    for w in weights:
        if w == 0.0:
            continue
        if not (w > 0) or math.isinf(w):
            return False
        fr, ex = math.frexp(w)
        m, e = int(math.ldexp(fr, 53)), ex - 53
        while m % 2 == 0:
            m //= 2
            e += 1
        parts.append((m, e))
    if not parts:
        return True
    q = min(e for _, e in parts)
    return sum(m << (e - q) for m, e in parts) * n_entries < 2 ** 53


class RefList:
    """points_of_interest (P x 5) and the weight classes as the library numbers them."""

    def __init__(self, pts, weights, nx=NX, ny=NY, dx=DX, dy=DY):
        self.pts = np.asarray(pts, dtype=np.float64).reshape(-1, 5)
        self.weights = list(weights)
        self.nx, self.ny, self.dx, self.dy = nx, ny, dx, dy

    # the setters
    @classmethod
    def set_points(cls, pts, **kw):
        pts = np.asarray(pts, dtype=np.float64).reshape(-1, 5)
        ws = []
        for w in pts[:, 3]:
            if w not in ws:
                ws.append(float(w))
        dx, dy = kw.get("dx", DX), kw.get("dy", DY)
        return cls(pts, ws or [dx * dy], **kw)

    @classmethod
    def grid_full(cls, orc, nx=NX, ny=NY, dx=DX, dy=DY):
        return cls(orc.createPOI(dx, dy, float(nx), float(ny)), [dx * dy], nx, ny, dx, dy)

    @classmethod
    def grid_bits(cls, mask, w):
        c = createpoi_cells(NX, NY)
        return cls(rows(c[mask[c]], w), [w])

    @classmethod
    def grid_cells(cls, mult, kls, cw):
        c = createpoi_cells(NX, NY)
        c = np.repeat(c, mult[c])                       # mult[c] copies of a cell next to each other
        pts = rows(c, 0.0)
        pts[:, 3] = np.asarray(cw, dtype=np.float64)[kls[c]]
        return cls(pts, cw)

    @classmethod
    def fire_init(cls, state, push_initial):
        c = createpoi_cells(NX, NY)
        return cls(rows(c[state[c] == 2] if push_initial else [], W), [W])

    # the changes
    def add(self, new):
        new = np.asarray(new, dtype=np.float64).reshape(-1, 5)
        if len(self.pts) == 0 and len(new):  # an empty store has no weight yet: the numbering restarts
            self.weights = []
        for w in new[:, 3]:
            if w not in self.weights:
                self.weights.append(float(w))
        self.pts = np.concatenate([self.pts, new])

    def remove(self, orc, discs):
        self.pts = orc.rmvCoveredPOI(discs, self.pts)

    # what the store must report
    def cells(self):
        i = np.rint((self.pts[:, 0] + self.dx / 2) / self.dx).astype(np.int64) - 1
        j = np.rint((self.pts[:, 1] + self.dy / 2) / self.dy).astype(np.int64) - 1
        return i + self.nx * j

    def hist(self):
        return np.bincount(self.cells(), minlength=self.nx * self.ny)

    def class_of(self):
        return np.array([self.weights.index(w) for w in self.pts[:, 3]], dtype=np.int32)

    def planes(self):
        """Bit planes the store needs: per class, the set bits of its cells' multiplicities (the kernels sweep 8)."""
        h, k = self.hist(), np.full(self.nx * self.ny, -1)
        k[self.cells()] = self.class_of()
        return sum(bin(int(np.bitwise_or.reduce(h[k == c], initial=0))).count("1") for c in range(len(self.weights)))

    def cell_weight(self):
        """cell -> weight of its entries (NaN where empty)."""
        cw = np.full(self.nx * self.ny, np.nan)
        cw[self.cells()] = self.pts[:, 3]
        return cw


# ---------------------------------------------------------------- CPU: the model against the oracle
def test_createpoi_order_is_the_oracles(orc):
    for nx, ny, dx, dy in ((NX, NY, DX, DY), (7, 5, 2.5, 4.0), (1, 9, 1.0, 3.0), (33, 2, 0.75, 5.0)):
        assert np.array_equal(rows(createpoi_cells(nx, ny), dx * dy, nx, dx, dy), orc.createPOI(dx, dy, nx, ny))
        assert np.array_equal(RefList.grid_full(orc, nx, ny, dx, dy).pts, orc.createPOI(dx, dy, nx, ny))


def test_grid_cells_expansion_and_removal_keep_list_order(orc):
    rng = np.random.default_rng(1)
    mult = rng.integers(0, 4, NX * NY)
    kls = rng.integers(0, 2, NX * NY)
    m = RefList.grid_cells(mult, kls, [W, H])
    full = orc.createPOI(DX, DY, NX, NY)
    k = np.repeat(np.arange(len(full)), mult[createpoi_cells(NX, NY)])
    assert np.array_equal(m.pts[:, :2], full[k, :2])
    assert np.array_equal(m.hist(), mult)
    assert np.array_equal(m.pts[:, 3], np.where(kls[m.cells()] == 0, W, H))
    discs = np.array([60.0, 130.0, 100.0, 95.0, 30.0, 22.0])
    keep = np.ones(len(m.pts), dtype=bool)
    for c in range(2):
        ax, ay = m.pts[:, 0] - discs[c], m.pts[:, 1] - discs[2 + c]
        keep &= ~(np.sqrt(ax * ax + ay * ay) < discs[4 + c])
    assert 0 < keep.sum() < len(keep)
    got = orc.rmvCoveredPOI(discs, m.pts)
    assert np.array_equal(got, m.pts[keep])         # the rest in its order
    # every entry of a covered cell goes: removal empties cells, never thins them
    left = np.bincount(RefList(got, [W, H]).cells(), minlength=NX * NY)
    assert np.all((left == 0) | (left == mult))


def test_one_class_block_order_does_not_change_the_area(orc):
    """What lets the model skip ordering the fire_init and fire_step blocks: inside a block of one weight the
    order of the entries cannot change calculateArea -- and across two classes it does (else nothing is tested)."""
    rng = np.random.default_rng(2)
    X = cands(rng, 64)
    for w in (W, H):
        block = rows(rng.integers(0, NX * NY, 900), w)
        tail = rows(rng.integers(0, NX * NY, 300), H2)
        for before, after in (([], []), ([], [tail]), ([tail], [])):
            lst = np.concatenate(before + [block] + after)
            base = [orc.calculateArea(x, lst)[0] for x in X]
            for _ in range(3):
                sh = np.concatenate(before + [block[rng.permutation(len(block))]] + after)
                assert [orc.calculateArea(x, sh)[0] for x in X] == base
    mixed = np.concatenate([rows(rng.integers(0, NX * NY, 600), H2), rows(rng.integers(0, NX * NY, 600), H)])
    sh = mixed[rng.permutation(len(mixed))]
    assert any(orc.calculateArea(x, mixed)[0] != orc.calculateArea(x, sh)[0] for x in X)


def test_area_exact_rule_restated():
    assert area_exact_rule([2.0 ** 30, 2.0 ** -16], 127) and not area_exact_rule([2.0 ** 30, 2.0 ** -16], 128)
    assert area_exact_rule([W], 10 ** 12) and not area_exact_rule([W, H], 2)
    assert area_exact_rule([H], 1) and area_exact_rule([0.0, W], 5)
    assert not area_exact_rule([W, -W], 1) and not area_exact_rule([W, math.inf], 1)


# ---------------------------------------------------------------- GPU helpers
def cands(rng, B, n=N, centre=100.0, spread=45.0):
    """Discs around the middle of the grid; the first half at R = r_max (no penalty, so the last bits of the area
    reach the objective), the rest with R an integer below it."""
    xy = centre + (rng.random((B, 2 * n)) * 2 - 1) * spread
    R = np.where(np.arange(B)[:, None] < B // 2, 36.0, rng.integers(6, 36, (B, n)).astype(np.float64))
    return np.rint(np.concatenate([xy, R], axis=1))


def same_bits(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def first_diff(a, b):
    d = np.flatnonzero(np.asarray(a).view(np.uint64) != np.asarray(b).view(np.uint64))
    return (int(d[0]), a[d[0]], b[d[0]]) if len(d) else None


class Checker:
    """After every operation: the store's statistics and the evaluation against the oracle on the model's list."""

    def __init__(self, cov, orc, X, r_max=R_MAX, **cons):
        self.cov, self.orc, self.X, self.r_max, self.cons = cov, orc, X, r_max, cons
        self.order_visible = 0  # checks where the order-free sum sum_k w_k count_k misses the oracle

    def __call__(self, eng, m, what=""):
        n = self.X.shape[1] // 3
        assert np.array_equal(eng.grid_cells(), m.hist()), what
        info = eng.grid_info()
        assert (info["n_entries"], info["n_cells"], info["n_classes"]) == \
            (len(m.pts), int((m.hist() > 0).sum()), len(m.weights)), what
        assert eng.class_weights() == m.weights, what
        assert info["area_exact"] == int(area_exact_rule(m.weights, len(m.pts))), what
        got = eng.eval_batch(self.X, want_class_count=True, want_progressive=True)
        if not info["area_exact"]:
            assert eng.last_launch()["kernel"] == ORDERED, what
        want = self.orc.eval_batch(self.X, n, self.r_max, m.pts, want_prog=True, **self.cons)
        assert np.array_equal(got["count"], want["count"]), what
        assert np.array_equal(got["feasible"], want["feasible"]), what
        assert same_bits(got["obj"], want["obj"]), (what, first_diff(got["obj"], want["obj"]))
        assert same_bits(got["progressive"], want["progressive"]), what
        k = m.class_of()
        for b in range(len(self.X)):
            assert got["class_count"][b].tolist() == self.orc.class_counts(self.X[b], m.pts, k, len(m.weights)).tolist(), (what, b)
        with np.errstate(invalid="ignore"):  # an infinite weight times a zero count
            naive = -(np.asarray(m.weights) * got["class_count"]).sum(axis=1) + \
                1e5 * np.abs(self.X[:, 2 * n:] - self.r_max).sum(axis=1)
        self.order_visible += int((naive != want["obj"]).any())
        return got


def pick(m, rng, k, w, empty, window=(8, 32)):
    """k list entries of weight w on cells of the central window that are empty (empty=True) or hold entries of
    weight w (empty=False), each cell at most once while there are enough; None when there is no such cell."""
    cw = m.cell_weight()
    lo, hi = window
    ii, jj = np.meshgrid(np.arange(lo, hi), np.arange(lo, hi), indexing="ij")
    cand = (ii + NX * jj).ravel()
    ok = cand[np.isnan(cw[cand])] if empty else cand[cw[cand] == w]
    return rows(rng.choice(ok, k, replace=k > len(ok)), w) if len(ok) else None


def mask_to_bits(mask):
    bits = np.zeros((NY, (NX + 31) // 32), dtype=np.uint32)
    for c in np.flatnonzero(mask):
        i, j = c % NX, c // NX
        bits[j, i // 32] |= np.uint32(1 << (i % 32))
    return bits


def fire_state(rng):
    state = np.where(rng.random(NX * NY) < 0.1, 0, 1).astype(np.uint8)
    for i in range(17, 23):
        for j in range(18, 22):
            state[i + NX * j] = 2
    return state


REMOVE_A = np.array([100.0, 100.0, 28.0])
REMOVE_B = np.array([80.0, 125.0, 110.0, 90.0, 14.0, 17.0])


def fire_steps(eng, orc, m, chk, state, first, count, seed=2026):
    for step in range(first, first + count):
        pushed = eng.fire_step(*WIND, seed, step, append=True)
        state, new = orc.fire_step(state, NX, NY, DX, DY, *WIND, step, seed)
        assert pushed == len(new)
        m.add(new)
        assert np.array_equal(eng.fire_state(), state)
        chk(eng, m, f"fire step {step}")
    return state


# ---------------------------------------------------------------- scripted lifecycles
def lc_points(eng, orc, chk, rng):
    full = orc.createPOI(DX, DY, NX, NY)
    full[(full[:, 0] > 90) & (full[:, 1] > 95), 3] = H
    m = RefList.set_points(full)
    eng.set_points(full, NX, NY, DX, DY)
    chk(eng, m, "set_points")
    for discs in (REMOVE_A, REMOVE_B):
        eng.remove_covered(discs)
        m.remove(orc, discs)
        chk(eng, m, "remove")
        new = np.concatenate([pick(m, rng, 40, H, True), pick(m, rng, 30, W, False), pick(m, rng, 20, H, False)])
        eng.add_points(new)
        m.add(new)
        chk(eng, m, "add")
    return m


def lc_full(eng, orc, chk, rng):
    m = RefList.grid_full(orc)
    eng.set_grid_full(NX, NY, DX, DY)
    chk(eng, m, "set_grid_full")
    eng.remove_covered(REMOVE_A)
    m.remove(orc, REMOVE_A)
    chk(eng, m, "remove")
    new = np.concatenate([pick(m, rng, 60, H, True), pick(m, rng, 40, W, False)])
    new = new[rng.permutation(len(new))]
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "add onto a createPOI store")
    eng.remove_covered(REMOVE_B)
    m.remove(orc, REMOVE_B)
    chk(eng, m, "remove")
    new = np.concatenate([pick(m, rng, 30, W, False), pick(m, rng, 30, H, True), pick(m, rng, 10, H, False)])
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "add")
    return m


def lc_bits(eng, orc, chk, rng):
    mask = rng.random(NX * NY) < 0.5
    eng.set_grid_bits(mask_to_bits(mask), NX, NY, DX, DY, weight=W)
    m = RefList.grid_bits(mask, W)
    chk(eng, m, "set_grid_bits")
    new = np.concatenate([pick(m, rng, 50, H, True), pick(m, rng, 50, W, False)])
    new = new[rng.permutation(len(new))]
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "add onto a bit grid")
    return m


def lc_cells(eng, orc, chk, rng):
    mult = rng.integers(0, 3, NX * NY).astype(np.uint8)
    kls = (rng.random(NX * NY) < 0.3).astype(np.uint8)
    eng.set_grid_cells(mult, NX, NY, DX, DY, cls=kls, class_weight=[W, H])
    m = RefList.grid_cells(mult, kls, [W, H])
    chk(eng, m, "set_grid_cells (the createPOI-order prefix)")
    new = np.concatenate([pick(m, rng, 30, H, False), pick(m, rng, 30, W, False), pick(m, rng, 20, H2, True)])
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "add")
    eng.remove_covered(REMOVE_A)
    m.remove(orc, REMOVE_A)
    chk(eng, m, "remove")
    new = np.concatenate([pick(m, rng, 30, H, True), pick(m, rng, 20, H2, False)])
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "add")
    return m


def lc_fire(eng, orc, chk, rng):
    cov = chk.cov
    state = fire_state(rng)
    eng.fire_init(state, NX, NY, DX, DY, push_initial=True)
    m = RefList.fire_init(state, True)
    chk(eng, m, "fire_init")
    state = fire_steps(eng, orc, m, chk, state, 1, 3)
    new = pick(m, rng, 60, H, True)
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "high weight onto cells that are not burning")
    before = eng.grid_cells()
    with pytest.raises(cov.CoverageError) as ei:
        eng.fire_step(*WIND, 2026, 4, append=True)
    assert ei.value.code == cov._lib.COV_ERR_STATE
    assert np.array_equal(eng.fire_state(), state) and np.array_equal(eng.grid_cells(), before)
    chk(eng, m, "after the refused fire step")
    eng.remove_covered(REMOVE_B)
    m.remove(orc, REMOVE_B)
    chk(eng, m, "remove")
    new = np.concatenate([pick(m, rng, 20, H, False), pick(m, rng, 20, W, False), pick(m, rng, 20, H, True)])
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "add")
    return m


def lc_fire_empty(eng, orc, chk, rng):
    state = fire_state(rng)
    eng.fire_init(state, NX, NY, DX, DY, push_initial=False)
    m = RefList.fire_init(state, False)
    chk(eng, m, "empty fire store")
    new = pick(m, rng, 50, H, True)
    eng.add_points(new)
    m.add(new)
    assert m.weights == [H]
    chk(eng, m, "first append names class 0")
    new = np.concatenate([pick(m, rng, 30, W, True), pick(m, rng, 30, H, False)])
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "second class")
    return m


def lc_emptied(eng, orc, chk, rng):
    m = lc_points(eng, orc, chk, rng)
    everything = np.array([100.0, 100.0, 1000.0])
    eng.remove_covered(everything)
    m.remove(orc, everything)
    assert len(m.pts) == 0
    chk(eng, m, "emptied")
    new = pick(m, rng, 40, H2, True)
    eng.add_points(new)
    m.add(new)
    assert m.weights == [H2]
    chk(eng, m, "numbering restarts")
    new = np.concatenate([pick(m, rng, 40, W, True), pick(m, rng, 20, H2, False)])
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "second class")
    return m


def lc_failed_append(eng, orc, chk, rng):
    cov = chk.cov
    m = RefList.grid_full(orc)
    eng.set_grid_full(NX, NY, DX, DY)
    eng.remove_covered(REMOVE_A)
    m.remove(orc, REMOVE_A)
    bad = np.concatenate([pick(m, rng, 20, H, True), rows([m.cells()[0]], H)])  # H onto a cell of weight 25
    with pytest.raises(cov.CoverageError) as ei:
        eng.add_points(bad)
    assert ei.value.code == cov._lib.COV_ERR_INVALID
    chk(eng, m, "after a refused append (mixed weights), no list given yet")
    new = pick(m, rng, 50, H, True)
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "add")
    c = int(m.cells()[-1])
    bad = np.concatenate([pick(m, rng, 10, W, False), rows(np.full(300, c), H)])  # > 255 entries on one cell
    with pytest.raises(cov.CoverageError) as ei:
        eng.add_points(bad)
    assert ei.value.code == cov._lib.COV_ERR_LIMIT
    chk(eng, m, "after a refused append (> 255 entries)")
    bad = rows([int(m.cells()[0])], H2)
    with pytest.raises(cov.CoverageError):
        eng.add_points(bad)
    chk(eng, m, "after a refused append (new weight on an occupied cell)")
    empty = int(np.flatnonzero(m.hist() == 0)[0])
    bad = np.concatenate([pick(m, rng, 10, H, False), rows(np.full(255, empty), H2)])
    after = RefList(m.pts, m.weights)
    after.add(bad)
    assert after.planes() > 8
    with pytest.raises(cov.CoverageError) as ei:  # 255 entries of a third class: 8 more bit planes
        eng.add_points(bad)
    assert ei.value.code == cov._lib.COV_ERR_LIMIT
    chk(eng, m, "after a refused append (more than 8 bit planes)")
    new = np.concatenate([pick(m, rng, 20, W, False), pick(m, rng, 20, H, False)])
    eng.add_points(new)
    m.add(new)
    chk(eng, m, "add")
    return m


LIFECYCLES = {"points": lc_points, "full": lc_full, "bits": lc_bits, "cells": lc_cells, "fire": lc_fire,
              "fire_empty": lc_fire_empty, "emptied": lc_emptied, "failed_append": lc_failed_append}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LIFECYCLES))
def test_lifecycle_list_order(cov, orc, engine, name):
    rng = np.random.default_rng(list(LIFECYCLES).index(name) + 100)
    X = cands(rng, 48)
    engine.set_params(N, R_MAX)
    chk = Checker(cov, orc, X)
    m = LIFECYCLES[name](engine, orc, chk, rng)
    assert len(m.weights) >= 2 and not area_exact_rule(m.weights, len(m.pts))
    assert chk.order_visible > 0  # the order-free sum misses the oracle somewhere: the order was under test


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [7, 8, 9])
def test_random_walk_list_order(cov, orc, engine, seed):
    """About 40 operations drawn from add (new or existing weight, onto empty or occupied cells), remove and fire
    step; the fire step is refused unless the store holds the one class of weight dx*dy."""
    rng = np.random.default_rng(seed)
    X = cands(rng, 32)
    engine.set_params(N, R_MAX)
    chk = Checker(cov, orc, X)
    state = fire_state(rng)
    engine.fire_init(state, NX, NY, DX, DY, push_initial=True)
    m = RefList.fire_init(state, True)
    chk(engine, m, "fire_init")
    ops = {"add": 0, "add refused": 0, "remove": 0, "fire": 0, "fire refused": 0}
    for step in range(1, 41):
        early = step <= 8  # the automaton runs while the store holds its one class
        op = rng.choice(["add", "remove", "fire", "fire"] if early else ["add", "add", "remove", "fire"])
        if op == "add":
            pool = list(m.weights) + [w for w in (H, H2, W) if w not in m.weights and len(m.weights) < 4]
            w = W if early else float(rng.choice(pool))
            k = int(rng.integers(1, 40))
            new = pick(m, rng, k, w, False) if rng.random() < 0.5 else None
            new = new if new is not None else pick(m, rng, k, w, True)
            if new is None:
                continue
            after = RefList(m.pts, m.weights)
            after.add(new)
            if after.planes() > 8:
                op = "add refused"
                with pytest.raises(cov.CoverageError) as ei:
                    engine.add_points(new)
                assert ei.value.code == cov._lib.COV_ERR_LIMIT
            else:
                engine.add_points(new)
                m.add(new)
        elif op == "remove":
            discs = np.concatenate([rng.uniform(40, 160, 2), rng.uniform(3, 25, 1)])
            engine.remove_covered(discs)
            m.remove(orc, discs)
        elif m.weights == [W]:
            pushed = engine.fire_step(*WIND, seed, step, append=True)
            state, new = orc.fire_step(state, NX, NY, DX, DY, *WIND, step, seed)
            assert pushed == len(new)
            m.add(new)
            assert np.array_equal(engine.fire_state(), state)
        else:
            op = "fire refused"
            with pytest.raises(cov.CoverageError) as ei:
                engine.fire_step(*WIND, seed, step, append=True)
            assert ei.value.code == cov._lib.COV_ERR_STATE
            assert np.array_equal(engine.fire_state(), state)
        ops[op] += 1
        chk(engine, m, f"op {step}: {op}")
    assert ops["add"] and ops["remove"] and ops["fire"]
    assert chk.order_visible > 0


# ---------------------------------------------------------------- every entry point on an order-sensitive store
class BorrowedEngine:
    """A CoverageEngine view of a handle the caller owns (a cov_multi shard)."""

    def __init__(self, cov, h):
        self.eng = cov.CoverageEngine.__new__(cov.CoverageEngine)
        self.eng._h, self.eng._pinned, self.eng.N, self.eng.device, self.eng.param_owner = C.c_void_p(h), [], None, 0, None

    def release(self):
        self.eng._h = None


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["full", "fire"])
def test_every_entry_point_on_order_sensitive_store(cov, orc, engine, name):
    lib = cov._lib.lib
    rng = np.random.default_rng(300)
    X = cands(rng, 200)
    B = len(X)
    cons = {"sep_min": 15.0}
    engine.set_params(N, R_MAX, sep_min=15.0)
    chk = Checker(cov, orc, X[:48], tan_half_fov=T, **cons)
    m = LIFECYCLES[name](engine, orc, chk, np.random.default_rng(7))
    assert engine.grid_info()["area_exact"] == 0
    want = orc.eval_batch(X, N, R_MAX, m.pts, **cons)
    assert (want["feasible"] == 0).any() and (want["feasible"] == 1).any()

    def same(got, what, sub=slice(None)):
        assert np.array_equal(got["count"], want["count"][sub]), what
        assert np.array_equal(got["feasible"], want["feasible"][sub]), what
        assert same_bits(got["obj"], want["obj"][sub]), (what, first_diff(got["obj"], want["obj"][sub]))

    def ordered(what):
        assert engine.last_launch()["kernel"] == ORDERED, what

    def winner(barrier, sub=slice(None)):
        o = np.where(want["feasible"][sub] == 1, want["obj"][sub], np.inf) if barrier else want["obj"][sub]
        return (float(o.min()), int(np.argmin(o))) if np.isfinite(o.min()) else (math.inf, -1)

    same(engine.eval_batch(X), "pageable")
    ordered("pageable")
    P = engine.pinned(X.shape)
    P[:] = X
    same(engine.eval_batch(P), "pinned")
    ordered("pinned")
    for zc in (0, 1):
        engine.set_option(cov.OPT_ZEROCOPY_OUT, zc)
        engine.set_option(cov.OPT_CHUNK, 32)  # several slices through the pipeline
        same(engine.eval_batch(X), f"chunked, zero-copy out {zc}")
        ordered("chunked")
        same(engine.eval_batch(P), f"pinned chunked, zero-copy out {zc}")
        engine.set_option(cov.OPT_CHUNK, 0)
        same(engine.eval_batch(P), f"pinned, zero-copy out {zc}")
    ex = engine.eval_batch(X, want_class_count=True, want_progressive=True)
    same(ex, "eval_batch_ex")
    for b in range(0, B, 9):
        assert ex["class_count"][b].tolist() == orc.class_counts(X[b], m.pts, m.class_of(), len(m.weights)).tolist()
    prog = orc.eval_batch(X, N, R_MAX, m.pts, want_prog=True)["progressive"]
    assert same_bits(ex["progressive"], prog)
    # device buffers
    dX, dO, dC, dF = (engine.device_alloc(n) for n in (X.nbytes, 8 * B, 8 * B, B))
    try:
        engine.memcpy_h2d(dX, np.ascontiguousarray(X))
        engine.eval_batch_device(dX, B, dO, dC, dF)
        got = {"obj": np.empty(B), "count": np.empty(B, dtype=np.int64), "feasible": np.empty(B, dtype=np.uint8)}
        engine.memcpy_d2h(got["obj"], dO)
        engine.memcpy_d2h(got["count"], dC)
        engine.memcpy_d2h(got["feasible"], dF)
        engine.sync()
        same(got, "eval_batch_device")
        ordered("eval_batch_device")
    finally:
        for p in (dX, dO, dC, dF):
            engine.device_free(p)
    for b in range(0, B, 13):
        assert same_bits([engine.eval_one(X[b])], [want["obj"][b]]), b
        ordered("eval_one")
    for barrier in (0, 1):
        assert engine.argmin(X, barrier=bool(barrier)) == winner(barrier), barrier
        ordered("argmin")
        best = engine.eval_batch_best(X, barrier=bool(barrier))
        same(best, "eval_batch_best")
        assert best["best"] == winner(barrier)
        ordered("eval_batch_best")
    # packed candidates (the candidates are integers)
    for dt in (np.int16, np.int32, np.float32):
        Q = cov.pack_candidates(X, 1.0, dt)
        same(engine.eval_batch_packed(Q, 1.0), f"packed {np.dtype(dt).name}")
        ordered("packed")
        for barrier in (False, True):
            r = engine.eval_batch_packed(Q, 1.0, best=True, barrier=barrier)
            same(r, f"packed {np.dtype(dt).name} with winner")
            assert r["best"] == winner(barrier)
    # a kernel choice does not override the list-order sum
    for k in (cov.KERNEL_SPAN, cov.KERNEL_SPAN_GENERAL, cov.KERNEL_BRUTE, cov.KERNEL_EXACT):
        engine.set_option(cov.OPT_KERNEL, k)
        same(engine.eval_batch(X), f"kernel option {k}")
        ordered(f"kernel option {k}")
    engine.set_option(cov.OPT_KERNEL, cov.KERNEL_AUTO)
    # native MADS: every returned objective is the reference's on the returned point
    for s in range(3):
        x, obj, _ = engine.mads_solve(X[s], n_iter=15, granularity=1.0, seed=s)
        if math.isfinite(obj):
            assert same_bits([obj], [orc.objective(x, R_MAX, m.pts)[0]]), s
    Xo, objs, _ = engine.mads_solve_batch(X[:24], n_iter=15, granularity=1.0, seed=5)
    fin = np.isfinite(objs)
    assert fin.any()
    for k in np.flatnonzero(fin):
        assert same_bits([objs[k]], [orc.objective(Xo[k], R_MAX, m.pts)[0]]), k
    # two handles of device 0 carried through the same lifecycle
    devs = (C.c_int * 2)(0, 0)
    mh = C.c_void_p()
    assert lib.cov_multi_create(devs, 2, C.byref(mh)) == 0
    shards = []
    try:
        for k in range(2):
            sh = BorrowedEngine(cov, lib.cov_multi_handle(mh, k))
            shards.append(sh)
            sh.eng.set_params(N, R_MAX, sep_min=15.0)
            mk = LIFECYCLES[name](sh.eng, orc, Checker(cov, orc, X[:8], tan_half_fov=T, **cons), np.random.default_rng(7))
            assert np.array_equal(mk.pts, m.pts)
        obj, cnt, fe = np.empty(B), np.empty(B, dtype=np.int64), np.empty(B, dtype=np.uint8)
        assert lib.cov_multi_eval_batch(mh, X.ctypes.data, B, obj.ctypes.data, cnt.ctypes.data, fe.ctypes.data) == 0
        same({"obj": obj, "count": cnt, "feasible": fe}, "cov_multi_eval_batch")
        for barrier in (0, 1):
            bo, bi = C.c_double(), C.c_int64()
            assert lib.cov_multi_argmin(mh, X.ctypes.data, B, barrier, C.byref(bo), C.byref(bi)) == 0
            assert (bo.value, bi.value) == winner(barrier)
    finally:
        for sh in shards:
            sh.release()
        lib.cov_multi_destroy(mh)


# ---------------------------------------------------------------- the ordered kernel at its edges
def edge_store(orc, rng, P):
    """P entries over the four classes W, H, 0.0, H2 (one weight per cell); a second copy of the first few cells
    at the end, so one cell sits at positions far apart."""
    cells = np.resize(rng.permutation(NX * NY), P)  # multiplicities 1-2: 2 planes per class, 8 in all
    ws = np.array([W, H, 0.0, H2])[cells % 4]
    pts = rows(cells, 0.0)
    pts[:, 3] = ws
    return pts


def edge_cands(rng, B, n):
    """Discs across and beyond the grid with R = 0, R = +Inf and off-grid centres mixed in."""
    xy = rng.uniform(-60, 260, (B, 2 * n))
    R = rng.uniform(0, 40, (B, n))
    R[rng.random((B, n)) < 0.15] = 0.0
    if B > 2:
        R[1, 0] = math.inf
        xy[2, :] = -500.0  # every disc off the grid
    return np.concatenate([xy, R], axis=1)


def ordered_vs_oracle(cov, orc, engine, m, X, n):
    engine.set_params(n, np.full(n, 30 * T))
    engine.set_option(cov.OPT_KERNEL, ORDERED)
    got = engine.eval_batch(X, want_class_count=True, want_progressive=True)
    assert engine.last_launch()["kernel"] == ORDERED
    want = orc.eval_batch(X, n, np.full(n, 30 * T), m.pts, want_prog=True)
    assert np.array_equal(got["count"], want["count"])
    assert same_bits(got["obj"], want["obj"]), first_diff(got["obj"], want["obj"])
    assert same_bits(got["progressive"], want["progressive"])
    k = m.class_of()
    for b in range(len(X)):
        assert got["class_count"][b].tolist() == orc.class_counts(X[b], m.pts, k, len(m.weights)).tolist(), b
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, 32, 33, 64, 1024])
def test_ordered_kernel_swarm_sizes(cov, orc, engine, n):
    rng = np.random.default_rng(n)
    pts = edge_store(orc, rng, 1500)
    engine.set_points(pts, NX, NY, DX, DY)
    m = RefList.set_points(pts)
    later = pts[:100]
    engine.add_points(later)
    m.add(later)
    assert m.weights == [float(w) for w in engine.class_weights()] and len(m.weights) == 4
    ordered_vs_oracle(cov, orc, engine, m, edge_cands(rng, 9 if n == 1024 else 40, n), n)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [0, 1, 31, 32, 33, 3000])
def test_ordered_kernel_list_lengths(cov, orc, engine, P):
    rng = np.random.default_rng(P + 1)
    pts = edge_store(orc, rng, P)
    engine.set_points(pts, NX, NY, DX, DY)
    m = RefList.set_points(pts)
    assert engine.grid_info()["n_entries"] == P
    got = ordered_vs_oracle(cov, orc, engine, m, edge_cands(rng, 40, 5), 5)
    assert P == 0 or got["count"][1] == P  # the R = +Inf disc covers every entry


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 7, 9, 1000])
def test_ordered_kernel_batch_sizes(cov, orc, engine, B):
    rng = np.random.default_rng(B + 2)
    pts = edge_store(orc, rng, 700)
    engine.set_points(pts, NX, NY, DX, DY)
    m = RefList.set_points(pts)
    ordered_vs_oracle(cov, orc, engine, m, edge_cands(rng, B, 5), 5)


@pytest.mark.gpu
@pytest.mark.parametrize("setter", ["cells", "full", "fire_init"])
def test_ordered_kernel_cross_check_dyadic(cov, orc, engine, setter):
    """COV_KERNEL_ORDERED on dyadic stores of every setter without a list: the same bits as the span kernels and
    the oracle on createPOI's order."""
    rng = np.random.default_rng(400)
    if setter == "cells":
        mult = rng.integers(0, 4, NX * NY).astype(np.uint8)
        kls = (rng.random(NX * NY) < 0.4).astype(np.uint8)
        engine.set_grid_cells(mult, NX, NY, DX, DY, cls=kls, class_weight=[W, 100.0])
        m = RefList.grid_cells(mult, kls, [W, 100.0])
    elif setter == "full":
        engine.set_grid_full(NX, NY, DX, DY)
        m = RefList.grid_full(orc)
    else:
        state = fire_state(rng)
        engine.fire_init(state, NX, NY, DX, DY, push_initial=True)
        m = RefList.fire_init(state, True)
    assert engine.grid_info()["area_exact"] == 1
    X = cands(rng, 300)
    engine.set_params(N, R_MAX)
    span = engine.eval_batch(X)
    assert engine.last_launch()["kernel"] != ORDERED
    engine.set_option(cov.OPT_KERNEL, ORDERED)
    got = engine.eval_batch(X)
    assert engine.last_launch()["kernel"] == ORDERED
    want = orc.eval_batch(X, N, R_MAX, m.pts)
    for r in (span, got):
        assert np.array_equal(r["count"], want["count"]) and same_bits(r["obj"], want["obj"])


# ---------------------------------------------------------------- the area_exact boundary
@pytest.mark.gpu
def test_area_exact_boundary(cov, orc, engine):
    """Weights 2^30 and 2^-16: odd mantissas 1 and 1 at exponents 30 and -16, so (2^46 + 1) * n_entries < 2^53
    holds up to 127 entries.  Below the bound the span kernels' sum_k w_k count_k is the list-order sum; above it the
    order matters and the ordered kernel must run."""
    A, b = 2.0 ** 30, 2.0 ** -16
    rng = np.random.default_rng(500)
    cells_a = rng.choice(NX * NY // 2, 126)          # duplicates allowed
    cell_b = NX * NY - 1
    pts = np.concatenate([rows(cells_a, A), rows([cell_b], b)])
    all_disc = [100.0, 100.0, 150.0]                 # covers the whole grid at R = r_max: obj = -area exactly
    X = np.array([all_disc] + [[x, y, 45.0] for x, y in rng.uniform(0, 200, (60, 2))])
    r_max = np.array([150.0])
    engine.set_points(pts, NX, NY, DX, DY)
    engine.set_params(1, r_max)
    chk = Checker(cov, orc, X, r_max=r_max)
    m = RefList.set_points(pts)
    steps = [("127 entries: below the bound", None), ("128: above", rows([cells_a[0]], A)),
             ("131", np.concatenate([rows([cells_a[1]], A), rows([cell_b, cell_b], b)]))]
    for what, new in steps:
        if new is not None:
            engine.add_points(new)
            m.add(new)
        info = engine.grid_info()
        assert info["area_exact"] == int(area_exact_rule(m.weights, len(m.pts))) == int(len(m.pts) <= 127), what
        got = chk(engine, m, what)
        assert (engine.last_launch()["kernel"] == ORDERED) == (len(m.pts) > 127), what
    # the order shows above the bound: 2^37 + 2^-16 rounds to 2^37 and the two later 2^-16 are lost one by one
    assert got["obj"][0] == -(2.0 ** 37) and -(A * 128 + b * 3) != got["obj"][0]
    assert chk.order_visible > 0
    for bad in (-W, math.inf):
        p2 = np.concatenate([rows(rng.choice(NX * NY // 2, 50), W), rows([cell_b], bad)])
        engine.set_points(p2, NX, NY, DX, DY)
        assert engine.grid_info()["area_exact"] == 0, bad
        chk(engine, RefList.set_points(p2), f"weight {bad}")
