"""GPU parity tests: libcoverage_cuda (through its C ABI, via ctypes) against the CPU oracle on the
same seeded inputs, the golden vectors, and size-independent properties at BASELINE's sizes.
Integer counts, feasibility flags and Float64 objectives are compared BIT-EXACTLY."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

T = math.tan((100 / 180 * math.pi) / 2)
KERNELS = {"span": 1, "span_general": 4, "brute": 2, "exact": 3}


def rand_candidates(rng, B, N, extent=500.0, hmin=5.0, hmax=30.0):
    return np.concatenate([rng.random((B, 2 * N)) * extent, (hmin + rng.random((B, N)) * (hmax - hmin)) * T], axis=1)


def same_doubles(a, b):
    """Bit-identical, except that any NaN equals any NaN (payloads are not part of the contract)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def check_against_oracle(cov, orc, eng, X, N, r_max, pts, **cons):
    want = orc.eval_batch(X, N, r_max, pts, want_prog=True, **cons)
    got = eng.eval_batch(X, want_progressive=True)
    assert np.array_equal(got["count"], want["count"]), np.flatnonzero(got["count"] != want["count"])[:10]
    assert np.array_equal(got["feasible"], want["feasible"])
    assert np.array_equal(got["obj"].view(np.uint64), want["obj"].view(np.uint64))
    assert np.array_equal(got["progressive"].view(np.uint64), want["progressive"].view(np.uint64))
    return got


# ---------------------------------------------------------------- golden vectors
def test_kat_static_grid(cov, orc, engine, kat):
    engine.set_grid_full(100, 100, 5.0, 5.0)
    info = engine.grid_info()
    assert (info["n_entries"], info["n_cells"], info["n_planes"], info["area_exact"]) == (10000, 10000, 1, 1)
    engine.set_params(1, [0.0], penalty_scale=0.0)
    for k in kat["kat2"]:
        r = engine.eval_batch(np.array([k["disc"]]))
        assert r["count"][0] == k["count"] and r["obj"][0] == -k["area"]
    r_max = np.array(kat["kat3"]["r_max"])
    engine.set_params(5, r_max)
    for name in ("kat3", "kat4"):
        k = kat[name]
        r = engine.eval_batch(np.array([k["x"]]))
        assert r["count"][0] == k["count"] and r["obj"][0] == k["objective"]
        assert engine.eval_one(k["x"]) == k["objective"]


def test_kat_static_grid_from_list(cov, orc, engine, kat):
    """Same vectors with the store built from the reference's own list layout (cov_set_points)."""
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    engine.set_points(pts, 100, 100, 5.0, 5.0)
    engine.set_params(5, kat["kat3"]["r_max"])
    X = np.array([kat["kat3"]["x"], kat["kat4"]["x"]])
    r = engine.eval_batch(X)
    assert r["count"].tolist() == [kat["kat3"]["count"], kat["kat4"]["count"]]
    assert r["obj"].tolist() == [kat["kat3"]["objective"], kat["kat4"]["objective"]]


def test_kat5_fire_list_multiplicities(cov, orc, engine, fire_rows, kat):
    k = kat["kat5"]
    allp = np.concatenate(fire_rows)
    engine.set_points(allp, 100, 100, 5.0, 5.0)
    info = engine.grid_info()
    assert (info["n_entries"], info["n_cells"]) == (k["entries"], k["unique"])
    assert info["n_planes"] == 2  # multiplicities 1..3 -> two bit planes
    mult = engine.grid_cells()
    assert np.bincount(mult)[1:].tolist() == [k["mult_hist"][str(m)] for m in (1, 2, 3)]
    engine.set_params(1, [0.0], penalty_scale=0.0)
    r = engine.eval_batch(np.array([k["all_covering_disc"]]))
    assert r["count"][0] == k["entries"] and r["obj"][0] == -25.0 * k["entries"]
    rng = np.random.default_rng(5)
    N = 5
    engine.set_params(N, np.full(N, 30 * T))
    X = rand_candidates(rng, 3000, N)
    X[:, N:2 * N] *= 0.75  # the fire sits at y < 355
    for name, kid in KERNELS.items():
        engine.set_option(cov.OPT_KERNEL, kid)
        got = check_against_oracle(cov, orc, engine, X, N, np.full(N, 30 * T), allp)
    assert got["count"].max() > 50


def test_recorded_targets(cov, orc, engine, targets):
    """Quadrotor_Targets.xlsx: recorded integer-valued MADS inputs of UAV 1 (x, y, z = R/tan)."""
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    engine.set_grid_full(100, 100, 5.0, 5.0)
    for key in ("root", "src"):
        t = targets[key]
        X = np.stack([t[:, 0], t[:, 1], t[:, 2] * T], axis=1)
        engine.set_params(1, [30 * T])
        check_against_oracle(cov, orc, engine, X, 1, [30 * T], pts)


# ---------------------------------------------------------------- randomised differential tests
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("force_exact", [0, 1])
def test_c1_random_vs_oracle(cov, orc, engine, kernel, force_exact):
    if kernel == "exact" and force_exact:
        pytest.skip("exact kernel has no FP32 stage")
    rng = np.random.default_rng(100 + force_exact)
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    engine.set_grid_full(100, 100, 5.0, 5.0)
    engine.set_option(cov.OPT_KERNEL, KERNELS[kernel])
    engine.set_option(cov.OPT_FORCE_EXACT, force_exact)
    N = 5
    r_max = np.full(N, 30 * T)
    X = rand_candidates(rng, 1500, N)
    X[:200] = np.rint(X[:200])           # integer mesh (granularity 1.0) -> many exact ties
    X[200:300, :2 * N] = np.rint(X[200:300, :2 * N] / 2.5) * 2.5  # centres on cell corners / centres
    X[200:300, 2 * N:] = np.rint(X[200:300, 2 * N:] / 2.5) * 2.5
    pre = X[7].copy()
    X[300:600] = pre + rng.normal(0, 4.0, (300, 3 * N))  # around the previous state: cons3 both ways
    engine.set_params(N, r_max, prev_xyR=pre, d_lim=10.0, tan_half_fov=T, sep_min=15.0, use_cons7=True)
    got = check_against_oracle(cov, orc, engine, X, N, r_max, pts, pre=pre, d_lim=10.0, tan_half_fov=T,
                               sep_min=15.0, use_cons7=True)
    assert 0 < got["feasible"].sum() < len(X)


def test_c2_fire_grid_vs_oracle(cov, orc, engine):
    n = 256
    d = 500.0 / n
    bits, nset = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    assert len(pts) == nset
    engine.set_grid_bits(bits, n, n, d, d)
    assert engine.grid_info()["n_entries"] == nset
    N = 5
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max)
    X = cov.synth.random_candidates(4096, N, seed=1)
    for name, kid in KERNELS.items():
        engine.set_option(cov.OPT_KERNEL, kid)
        check_against_oracle(cov, orc, engine, X[:4096 if name != "exact" else 512], N, r_max, pts)


def test_c3_shape_vs_oracle(cov, orc, engine):
    n = 1024
    d = 500.0 / n
    bits, nset = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    engine.set_grid_bits(bits, n, n, d, d)
    N = 50
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max, sep_min=15.0)
    X = cov.synth.random_candidates(96, N, seed=2)
    X[:8, :2 * N] = 100 + X[:8, :2 * N] * 0.1  # a tight swarm: heavy overlap, cons8 violated
    got = check_against_oracle(cov, orc, engine, X, N, r_max, pts, sep_min=15.0)
    engine.set_option(cov.OPT_KERNEL, KERNELS["brute"])
    check_against_oracle(cov, orc, engine, X[:32], N, r_max, pts, sep_min=15.0)
    assert got["count"].max() > 1000


def test_c4_shape_vs_oracle(cov, orc, engine):
    n = 4096
    d = 500.0 / n
    bits, nset = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    engine.set_grid_bits(bits, n, n, d, d)
    N = 200
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max, sep_min=15.0)
    X = cov.synth.random_candidates(6, N, seed=3)
    check_against_oracle(cov, orc, engine, X, N, r_max, pts, sep_min=15.0)


def test_near_boundary_adversarial(cov, orc, engine):
    """Centres placed so that the radicand of some cell is within a few ulps of T(R)."""
    rng = np.random.default_rng(42)
    n, d = 64, 500.0 / 64
    pts = orc.createPOI(d, d, float(n), float(n))
    engine.set_grid_full(n, n, d, d)
    rows = []
    for _ in range(1500):
        i, j = rng.integers(1, n + 1, 2)
        px, py = i * d - d / 2, j * d - d / 2
        R = float((5 + rng.random() * 25) * T) if rng.random() < 0.7 else float(rng.integers(4, 40))
        th = rng.random() * 2 * math.pi if rng.random() < 0.6 else rng.choice([0, math.pi / 2, math.pi])
        cx, cy = px - R * math.cos(th), py - R * math.sin(th)
        for _ in range(int(rng.integers(0, 4))):
            cx = math.nextafter(cx, cx + rng.choice([-1.0, 1.0]))
        rows.append([cx, cy, R])
    X = np.array(rows)
    for kernel in ("span", "span_general", "brute"):
        for fe in (0, 1):
            engine.set_option(cov.OPT_KERNEL, KERNELS[kernel])
            engine.set_option(cov.OPT_FORCE_EXACT, fe)
            engine.set_params(1, [30 * T])
            check_against_oracle(cov, orc, engine, X, 1, [30 * T], pts)


def test_non_f32_lattice_and_ragged_width(cov, orc, engine):
    """dx = 0.1 (not exactly representable), nx = 77 (ragged last word), ny = 45."""
    rng = np.random.default_rng(8)
    nx, ny, dx, dy = 77, 45, 0.1, 0.3
    fire = rng.random((nx, ny)) < 0.6
    bits = cov.synth.pack_bits(fire)
    pts = cov.synth.points_from_bits(bits, nx, dx, dy)
    engine.set_grid_bits(bits, nx, ny, dx, dy)
    N = 3
    X = np.concatenate([rng.random((800, N)) * 9 - 0.6, rng.random((800, N)) * 15 - 0.8,
                        rng.random((800, N)) * 2.5], axis=1)
    r_max = np.full(N, 1.0)
    for kernel in ("span", "span_general", "brute", "exact"):
        engine.set_option(cov.OPT_KERNEL, KERNELS[kernel])
        engine.set_params(N, r_max)
        check_against_oracle(cov, orc, engine, X, N, r_max, pts)


# ---------------------------------------------------------------- edge cases
def test_edge_radii_and_far_centres(cov, orc, engine):
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    engine.set_grid_full(100, 100, 5.0, 5.0)
    N = 2
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max)
    inf, nan = math.inf, math.nan
    X = np.array([
        [250, 250, 250, 250, 0.0, 0.0],            # R = 0: nothing covered
        [250, 250, 250, 250, -5.0, -0.0],          # negative R
        [250, 250, 250, 250, nan, 10.0],           # NaN R never covers, NaN penalty
        [250, 250, 250, 250, inf, 1.0],            # infinite R covers everything
        [-1e6, 250, 1e6, 250, 30.0, 30.0],         # far outside
        [1e300, 250, 250, -1e300, 1e300, 20.0],    # huge coordinates and radius (overflowing squares)
        [250, 1e18, 250, 250, 1e18, 3.0],          # absorption: |py - cy| rounds
        [2.5, 497.5, 2.5, 497.5, 2.5, 2.6],        # corner cells
        [250, 250, 250, 250, 1e-300, 5e-324],      # denormal radii
        [nan, 250, 250, 250, 10.0, 10.0],          # NaN centre
        [inf, 250, 250, 250, inf, 10.0],           # inf - inf = NaN in the radicand
        [0, 500, 0, 500, 707.2, 1.0],              # everything within one disc
    ], dtype=np.float64)
    for kernel in ("span", "span_general", "brute", "exact"):
        engine.set_option(cov.OPT_KERNEL, KERNELS[kernel])
        want = orc.eval_batch(X, N, r_max, pts, want_prog=True)
        for which in (0, 1, 2):  # cons1_progressive, then the single-UAV forms (src/TDM_Constraints.jl:182-221)
            engine.set_option(cov.OPT_PROGRESSIVE_INDEX, which)
            got = engine.eval_batch(X, want_progressive=True)
            assert np.array_equal(got["count"], want["count"]), (kernel, got["count"], want["count"])
            assert same_doubles(got["obj"], want["obj"]), (kernel, got["obj"], want["obj"])
            wp = want["progressive"] if which == 0 else np.array([orc.consK_progressive(x, r_max, which) for x in X])
            # NaN R of UAV 1 (row 2): Julia's max(NaN, 0.0) is NaN and the sum carries it; UAV 2 alone does not see it
            assert same_doubles(got["progressive"], wp), (kernel, which, got["progressive"], wp)
            assert np.isnan(wp[2]) == (which in (0, 1)) and wp[3] == (math.inf if which in (0, 1) else 0.0)
        engine.set_option(cov.OPT_PROGRESSIVE_INDEX, 0)
    engine.set_option(cov.OPT_PROGRESSIVE_INDEX, 3)  # UAV 3 of a 2-UAV swarm
    with pytest.raises(cov.CoverageError):
        engine.eval_batch(X, want_progressive=True)
    engine.set_option(cov.OPT_PROGRESSIVE_INDEX, 0)


def test_empty_inputs(cov, orc, engine):
    engine.set_points(np.zeros((0, 5)), 100, 100, 5.0, 5.0)
    info = engine.grid_info()
    assert info["n_entries"] == 0
    engine.set_params(5, np.full(5, 30 * T))
    X = cov.synth.random_candidates(64, 5, seed=4)
    r = engine.eval_batch(X)
    assert not r["count"].any()
    want = orc.eval_batch(X, 5, np.full(5, 30 * T), np.zeros((0, 5)))
    assert np.array_equal(r["obj"], want["obj"])
    r0 = engine.eval_batch(np.zeros((0, 15)))
    assert r0["obj"].shape == (0,)


def test_state_and_argument_errors(cov, engine):
    e = engine
    e.N = 1
    with pytest.raises(cov.CoverageError) as ei:
        e.eval_batch(np.zeros((1, 3)))
    assert ei.value.code == cov._lib.COV_ERR_STATE
    e.set_grid_full(10, 10, 5.0, 5.0)
    with pytest.raises(cov.CoverageError) as ei:
        e.eval_batch(np.zeros((1, 3)))
    assert ei.value.code == cov._lib.COV_ERR_STATE and "parameters" in ei.value.message
    with pytest.raises(cov.CoverageError) as ei:
        e.set_points(np.array([[2.6, 2.5, 25, 25, 0]]), 10, 10, 5.0, 5.0)
    assert ei.value.code == cov._lib.COV_ERR_OFF_LATTICE
    with pytest.raises(cov.CoverageError) as ei:
        e.set_points(np.array([[52.5, 2.5, 25, 25, 0]]), 10, 10, 5.0, 5.0)  # outside the lattice
    assert ei.value.code == cov._lib.COV_ERR_OFF_LATTICE
    with pytest.raises(cov.CoverageError) as ei:
        e.set_grid_full(0, 10, 5.0, 5.0)
    assert ei.value.code == cov._lib.COV_ERR_INVALID
    with pytest.raises(cov.CoverageError) as ei:
        e.set_grid_full(40000, 10, 5.0, 5.0)
    assert ei.value.code == cov._lib.COV_ERR_LIMIT
    with pytest.raises(cov.CoverageError):
        cov.CoverageEngine(9999)


# ---------------------------------------------------------------- cell store operations
def test_weight_classes_and_ordered_sum(cov, orc, engine, fire_rows):
    """High-interest weights (src/CellFunctions.jl:41-45): per-class integer counts are exact; the
    order-dependent Float64 area is replayed on the host from the device's covered mask."""
    allp = np.concatenate(fire_rows[:30]).copy()
    hi = (allp[:, 0] > 200) & (allp[:, 0] < 300) & (allp[:, 1] > 250)
    allp[hi, 3] = (30.0 * T) ** 2 * math.pi
    engine.set_points(allp, 100, 100, 5.0, 5.0)
    info = engine.grid_info()
    assert info["n_classes"] == 2 and info["area_exact"] == 0
    N = 4
    engine.set_params(N, np.full(N, 30 * T))
    rng = np.random.default_rng(21)
    X = rand_candidates(rng, 400, N)
    X[:, N:2 * N] = 200 + X[:, N:2 * N] * 0.3
    got = engine.eval_batch(X, want_class_count=True)
    first_w = allp[0, 3]
    class_of = (allp[:, 3] != first_w).astype(np.int32)
    for b in range(0, 400, 7):
        want = orc.class_counts(X[b], allp, class_of, 2)
        assert got["class_count"][b].tolist() == want.tolist()
    ACC = cov.AreaCoverageCalculation
    pl = ACC.PointList(allp, 100, 100, 5.0, 5.0)
    res = ACC.ResidentList(pl, engine=engine)
    for b in range(0, 400, 23):
        area, cnt, _ = orc.calculateArea(X[b], allp)
        assert ACC.calculateArea(X[b], res) == area
    obj = cov.TDM_STATIC_opt.createObjective(res, N, np.full(N, 30 * T))
    for b in range(0, 400, 57):
        assert obj(X[b]) == orc.objective(X[b], np.full(N, 30 * T), allp)[0]


def test_ordered_kernel_non_dyadic_weights_at_scale(cov, orc, engine, fire_rows):
    """Non-dyadic weights ((h_max tan(FOV/2))^2 pi, src/CellFunctions.jl:41-45): the Float64 area depends on the list
    order of the additions; the library replays it on the device (ordered kernel).  >= 10^4 candidates through
    obj.batch, bit for bit against the C restatement; then the list evolves (rmvCoveredPOI, update_POI's push!)."""
    allp = np.concatenate(fire_rows[:30]).copy()
    hi = (allp[:, 0] > 200) & (allp[:, 0] < 300) & (allp[:, 1] > 250)
    allp[hi, 3] = (30.0 * T) ** 2 * math.pi
    N = 4
    r_max = np.full(N, 30 * T)
    ACC = cov.AreaCoverageCalculation
    pl = ACC.PointList(allp, 100, 100, 5.0, 5.0)
    res = ACC.ResidentList(pl, engine=engine)
    obj = cov.TDM_STATIC_opt.createObjective(res, N, r_max)
    rng = np.random.default_rng(33)
    X = rand_candidates(rng, 12_000, N)
    X[:, N:2 * N] = 200 + X[:, N:2 * N] * 0.3
    got = obj.batch(X)
    assert engine.grid_info()["area_exact"] == 0 and engine.last_launch()["kernel"] == cov.KERNEL_ORDERED
    want = orc.eval_batch(X, N, r_max, allp)
    assert np.array_equal(got.view(np.uint64), want["obj"].view(np.uint64))
    full = engine.eval_batch(X[:3000], want_class_count=True)
    assert np.array_equal(full["count"], want["count"][:3000]) and full["class_count"].sum(axis=1).tolist() == want["count"][:3000].tolist()
    # the order-free formula would differ in the last bits for some candidates (else this test proves nothing)
    w = engine.class_weights()
    naive = -(w[0] * full["class_count"][:, 0] + w[1] * full["class_count"][:, 1]) + 1e5 * np.abs(X[:3000, 2 * N:] - r_max).sum(axis=1)
    assert (naive != want["obj"][:3000]).any()
    # the list evolves: removal keeps the order of the rest, appended entries go to the end
    discs = X[int(np.argmax(want["count"]))]
    ACC.rmvCoveredPOI(discs, res)
    now = orc.rmvCoveredPOI(discs, allp)
    assert np.array_equal(res.points.data, now)
    more = np.concatenate(fire_rows[30:34]).copy()
    more[::3, 3] = (30.0 * T) ** 2 * math.pi  # (one weight per cell: duplicates within these rows share it below)
    _, first = np.unique(more[:, :2], axis=0, return_index=True)
    keyw = {tuple(more[k, :2]): more[k, 3] for k in first}
    for q in range(len(more)):
        more[q, 3] = keyw[tuple(more[q, :2])]
    taken = {tuple(p[:2]): p[3] for p in now}
    more = more[[tuple(p[:2]) not in taken or taken[tuple(p[:2])] == p[3] for p in more]]
    res.points.append(more)
    engine.add_points(more)
    res.mark_synced()
    now = np.concatenate([now, more])
    got2 = obj.batch(X[:4000])
    want2 = orc.eval_batch(X[:4000], N, r_max, now)
    assert np.array_equal(got2.view(np.uint64), want2["obj"].view(np.uint64))
    assert obj(X[5]) == want2["obj"][5] and ACC.calculateArea(X[5], res) == orc.calculateArea(X[5], now)[0]


def test_ordered_kernel_as_cross_check(cov, orc, engine, fire_rows):
    """COV_KERNEL_ORDERED on dyadic stores: the reference's own loop over the list, against the oracle -- on the fire
    list (duplicates) and on a bit grid, where no list was given and the order is createPOI's."""
    pts = np.concatenate(fire_rows[:20])
    engine.set_points(pts, 100, 100, 5.0, 5.0)
    N = 5
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max, sep_min=15.0)
    engine.set_option(cov.OPT_KERNEL, cov.KERNEL_ORDERED)
    rng = np.random.default_rng(34)
    X = rand_candidates(rng, 3000, N)
    X[:, N:2 * N] = 200 + X[:, N:2 * N] * 0.3
    check_against_oracle(cov, orc, engine, X, N, r_max, pts, sep_min=15.0)
    assert engine.last_launch()["kernel"] == cov.KERNEL_ORDERED
    n, d = 256, 500.0 / 256
    bits, _ = cov.synth.fire_grid(n)
    engine.set_grid_bits(bits, n, n, d, d)
    engine.set_params(N, r_max, sep_min=15.0)
    check_against_oracle(cov, orc, engine, cov.synth.random_candidates(300, N, seed=5), N, r_max,
                         cov.synth.points_from_bits(bits, n, d, d), sep_min=15.0)


def test_remove_covered_and_add_points(cov, orc, engine, fire_rows):
    pts = np.concatenate(fire_rows[:10])
    engine.set_points(pts, 100, 100, 5.0, 5.0)
    discs = np.array([220.0, 260.0, 345.0, 340.0, 12.0, 14.0])
    want = orc.rmvCoveredPOI(discs, pts)
    removed = engine.remove_covered(discs)
    assert removed == len(pts) - len(want)
    mult = engine.grid_cells()
    ref = np.zeros(100 * 100, dtype=np.int64)
    pl = cov.AreaCoverageCalculation.PointList(want, 100, 100, 5.0, 5.0)
    np.add.at(ref, pl.cell_index(), 1)
    assert np.array_equal(mult, ref)
    engine.add_points(fire_rows[10])
    ref2 = ref.copy()
    np.add.at(ref2, cov.AreaCoverageCalculation.PointList(fire_rows[10], 100, 100, 5.0, 5.0).cell_index(), 1)
    assert np.array_equal(engine.grid_cells(), ref2)
    assert engine.grid_info()["n_entries"] == len(want) + len(fire_rows[10])
    # and the objective sees the updated store
    now = np.concatenate([want, fire_rows[10]])
    N = 3
    engine.set_params(N, np.full(N, 30 * T))
    rng = np.random.default_rng(9)
    X = rand_candidates(rng, 500, N)
    X[:, N:2 * N] = 250 + X[:, N:2 * N] * 0.25
    check_against_oracle(cov, orc, engine, X, N, np.full(N, 30 * T), now)


def test_covered_mask(cov, orc, engine):
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    engine.set_grid_full(100, 100, 5.0, 5.0)
    engine.set_params(2, [0.0, 0.0])
    x = np.array([100.3, 300.7, 200.1, 50.9, 33.3, 17.2])
    mask = engine.covered_mask(x).astype(bool)
    pl = cov.AreaCoverageCalculation.PointList(pts, 100, 100, 5.0, 5.0)
    kept = orc.rmvCoveredPOI(x, pts)
    assert (~mask[pl.cell_index()]).sum() == len(kept)


def test_argmin_and_barrier(cov, orc, engine):
    engine.set_grid_full(100, 100, 5.0, 5.0)
    N = 5
    r_max = np.full(N, 30 * T)
    rng = np.random.default_rng(77)
    pre = rand_candidates(rng, 1, N)[0]
    X = pre + rng.normal(0, 3.5, (5000, 3 * N))
    engine.set_params(N, r_max, prev_xyR=pre, d_lim=10.0, tan_half_fov=T)
    r = engine.eval_batch(X)
    feas = r["feasible"].astype(bool)
    assert 0 < feas.sum() < len(X)
    bo, bi = engine.argmin(X, barrier=True)
    masked = np.where(feas, r["obj"], np.inf)
    assert bi == int(np.argmin(masked)) and bo == masked[bi]
    bo2, bi2 = engine.argmin(X, barrier=False)
    assert bi2 == int(np.argmin(r["obj"])) and bo2 == r["obj"][bi2]
    engine.set_params(N, r_max, prev_xyR=pre + 1000.0, d_lim=10.0, tan_half_fov=T)
    bo3, bi3 = engine.argmin(X, barrier=True)
    assert bi3 == -1 and bo3 == math.inf


# ---------------------------------------------------------------- host-side mirror of the reference API
def test_reference_api_static(cov, orc, kat):
    CF, ACC, OPT, TC = cov.CellFunctions, cov.AreaCoverageCalculation, cov.TDM_STATIC_opt, cov.TDM_Constraints
    cells = CF.initialise_POI(CF.Cells(), "static")
    assert len(cells.points_of_interest) == 10000
    r_max = np.array(kat["kat3"]["r_max"])
    obj = OPT.createObjective(cells, 5, r_max)
    assert obj(np.array(kat["kat3"]["x"])) == kat["kat3"]["objective"]
    assert obj(np.array(kat["kat4"]["x"])) == kat["kat4"]["objective"]
    assert ACC.calculateArea(np.array(kat["kat4"]["x"]), cells.points_of_interest) == kat["kat4"]["area"]
    X = np.array([kat["kat3"]["x"], kat["kat4"]["x"]])
    assert obj.batch(X).tolist() == [kat["kat3"]["objective"], kat["kat4"]["objective"]]
    # r_max is captured by reference (mutated between timesteps, src/FullSimulation.jl:65-76)
    r_max[0] = 15 * T
    assert obj(np.array(kat["kat4"]["x"])) == orc.objective(kat["kat4"]["x"], r_max, cells.points_of_interest.data)[0]
    # rmvCoveredPOI then the objective again
    discs = np.array(kat["kat4"]["x"])
    want = orc.rmvCoveredPOI(discs, cells.points_of_interest.data)
    cells = CF.rmvCoveredPOI(cells, discs)
    assert np.array_equal(cells.points_of_interest.data, want)
    x5 = discs.copy()
    x5[:5] += 20
    assert obj(x5) == orc.objective(x5, r_max, want)[0]
    # constraints
    pre = ACC.make_circles(discs)
    cons3 = TC.create_cons3(pre, 100 / 180 * math.pi, 10 * np.ones(5))
    rng = np.random.default_rng(3)
    Xc = discs + rng.normal(0, 4, (300, 15))
    assert cons3.batch(Xc).tolist() == [orc.cons3(x, discs, T, np.full(5, 10.0)) for x in Xc]
    assert cons3(discs) is True and TC.cons1(discs) is True
    cons8 = TC.create_cons8(5)
    assert cons8.batch(Xc).tolist() == [orc.cons8(x) for x in Xc]
    cons7 = TC.create_cons7(5, 100 / 180 * math.pi)
    Xc[:, 5:10] -= 60
    assert cons7.batch(Xc).tolist() == [orc.cons7(x, T) for x in Xc]
    prog = TC.create_cons1_progressive(5, r_max)
    assert prog.batch(Xc).tolist() == [orc.cons1_progressive(x, r_max) for x in Xc]
    Xp = Xc.copy()
    Xp[:, 10:] += rng.normal(0, 30, (300, 5))  # radii on both sides of r_max
    prog2, prog3 = TC.create_cons2_progressive(5, r_max), TC.create_cons3_progressive(5, r_max)
    assert prog2.batch(Xp).tolist() == [orc.consK_progressive(x, r_max, 2) for x in Xp]  # src/TDM_Constraints.jl:197-208
    assert prog3.batch(Xp).tolist() == [orc.consK_progressive(x, r_max, 3) for x in Xp]  # :210-221
    assert prog.batch(Xp).tolist() == [orc.cons1_progressive(x, r_max) for x in Xp]      # and back to the sum
    assert prog2(Xp[0]) == orc.consK_progressive(Xp[0], r_max, 2) and (prog2.batch(Xp) > 0).any()
    with pytest.raises(ValueError):
        TC.create_cons3_progressive(2, r_max[:2])
    # fused constraints
    rest = obj.fuse([TC.cons1, cons3, lambda x: True])
    assert len(rest) == 1
    o, f = obj.batch(Xc, want_feasible=True)
    assert f.tolist() == [orc.cons3(x, discs, T, np.full(5, 10.0)) for x in Xc]
    cells.close()


def test_reference_api_dynamic(cov, orc, fire_rows):
    CF, OPT = cov.CellFunctions, cov.TDM_STATIC_opt
    cells = CF.initialise_POI(CF.Cells(), "dynamic", fire_rows=fire_rows)
    ref = np.concatenate(fire_rows[:10])
    assert np.array_equal(cells.points_of_interest.data, ref)
    N = 5
    r_max = np.full(N, 30 * T)
    rng = np.random.default_rng(31)
    discs = np.concatenate([200 + rng.random(N) * 100, 300 + rng.random(N) * 50, np.full(N, 10 * T)])
    for t in range(1, 8):
        cells = CF.update_POI(cells, t)
        if t != 1:
            ref = np.concatenate([ref, fire_rows[t + 10 - 1]])
        cells = CF.rmvCoveredPOI(cells, discs)
        ref = orc.rmvCoveredPOI(discs, ref)
        assert np.array_equal(cells.points_of_interest.data, ref)
        obj = OPT.createObjective(cells, N, r_max)
        X = discs + rng.normal(0, 6, (64, 3 * N))
        want = orc.eval_batch(X, N, r_max, ref)["obj"]
        assert np.array_equal(obj.batch(X), want)
        assert obj(X[0]) == want[0]
        discs = X[int(np.argmin(want))]
    cells.close()


# ---------------------------------------------------------------- device-resident path, pipeline, multi-GPU
def test_device_path_and_generator(cov, orc, engine):
    n = 256
    d = 500.0 / n
    bits, _ = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    engine.set_grid_bits(bits, n, n, d, d)
    N, B = 5, 5000
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max)
    dX = engine.device_alloc(B * 3 * N * 8)
    d_obj, d_cnt, d_fe = engine.device_alloc(B * 8), engine.device_alloc(B * 8), engine.device_alloc(B)
    engine.generate_candidates(dX, B, N, seed=2026, first_index=123456789012)
    X = np.empty((B, 3 * N))
    engine.memcpy_d2h(X, dX)
    engine.sync()
    assert np.array_equal(X, cov.synth.philox_candidates(B, N, 2026, 123456789012))
    engine.eval_batch_device(dX, B, d_obj, d_cnt, d_fe)
    obj, cnt = np.empty(B), np.empty(B, dtype=np.int64)
    engine.memcpy_d2h(obj, d_obj)
    engine.memcpy_d2h(cnt, d_cnt)
    engine.sync()
    assert engine.last_kernel_ms() > 0
    want = orc.eval_batch(X, N, r_max, pts)
    assert np.array_equal(cnt, want["count"]) and np.array_equal(obj, want["obj"])
    for p in (dX, d_obj, d_cnt, d_fe):
        engine.device_free(p)


def test_host_pipeline_chunks_and_pinned(cov, orc, engine):
    engine.set_grid_full(100, 100, 5.0, 5.0)
    N, B = 5, 20000
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max)
    X = cov.synth.random_candidates(B, N, seed=5)
    base = engine.eval_batch(X)
    for chunk in (1, 999, 4096):
        if chunk == 1:
            sub = engine.eval_batch(X[:50])
            engine.set_option(cov.OPT_CHUNK, 1)
            r = engine.eval_batch(X[:50])
            assert np.array_equal(r["obj"], sub["obj"])
            continue
        engine.set_option(cov.OPT_CHUNK, chunk)
        r = engine.eval_batch(X)
        for k in ("obj", "count", "feasible"):
            assert np.array_equal(r[k], base[k])
    Xp = engine.pinned((B, 3 * N))
    Xp[:] = X
    out = {"obj": engine.pinned((B,)), "count": engine.pinned((B,), np.int64), "feasible": engine.pinned((B,), np.uint8)}
    r = engine.eval_batch(Xp, out=out)           # pinned buffers through the slice pipeline (OPT_CHUNK still set)
    for k in ("obj", "count", "feasible"):
        assert np.array_equal(r[k], base[k])
    engine.set_option(cov.OPT_CHUNK, 0)
    for zc in (1, 0):                              # one zero-copy launch on the caller's buffers / copy engines
        engine.set_option(cov.OPT_ZEROCOPY_OUT, zc)
        for k in out:
            out[k][:] = 0
        r = engine.eval_batch(Xp, out=out)
        for k in ("obj", "count", "feasible"):
            assert np.array_equal(r[k], base[k]), (zc, k)
        for nb in (1, 30, 700, 2184):              # the small-batch path: pinned scratch, zero-copy or copied
            r = engine.eval_batch(X[:nb])
            for k in ("obj", "count", "feasible"):
                assert np.array_equal(r[k], base[k][:nb]), (zc, nb, k)
    engine.set_option(cov.OPT_ZEROCOPY_OUT, 1)
    sample = orc.eval_batch(X[:300], N, r_max, orc.createPOI(5.0, 5.0, 100.0, 100.0))
    assert np.array_equal(base["obj"][:300], sample["obj"])


@pytest.mark.parametrize("spread", [False, True])
def test_multi_shards(cov, orc, spread):
    """cov_multi: contiguous shards, host gather.  spread=False: two handles on device 0 (always runs);
    spread=True: one handle per visible GPU (needs >= 2 devices, e.g. gpurun --gpus 2)."""
    import ctypes as C
    lib = cov._lib.lib
    ndev = cov.device_count()
    if spread and ndev < 2:
        pytest.skip("needs at least two CUDA devices")
    ids = list(range(ndev)) if spread else [0, 0]
    devs = (C.c_int * len(ids))(*ids)
    m = C.c_void_p()
    assert lib.cov_multi_create(devs, len(ids), C.byref(m)) == 0
    try:
        N, B = 5, 3001
        r_max = np.full(N, 30 * T)
        for k in range(lib.cov_multi_size(m)):
            h = lib.cov_multi_handle(m, k)
            assert lib.cov_set_grid_full(h, 100, 100, 5.0, 5.0) == 0
            assert lib.cov_set_params(h, N, r_max.ctypes.data, 1e5, None, None, T, 0.0, 0) == 0
        X = cov.synth.random_candidates(B, N, seed=6)
        obj, cnt, fe = np.empty(B), np.empty(B, dtype=np.int64), np.empty(B, dtype=np.uint8)
        assert lib.cov_multi_eval_batch(m, X.ctypes.data, B, obj.ctypes.data, cnt.ctypes.data, fe.ctypes.data) == 0
        want = orc.eval_batch(X, N, r_max, orc.createPOI(5.0, 5.0, 100.0, 100.0))
        assert np.array_equal(obj, want["obj"]) and np.array_equal(cnt, want["count"])
        bo, bi = C.c_double(), C.c_int64()
        assert lib.cov_multi_argmin(m, X.ctypes.data, B, 1, C.byref(bo), C.byref(bi)) == 0
        assert bi.value == int(np.argmin(obj)) and bo.value == obj.min()
    finally:
        lib.cov_multi_destroy(m)


# ---------------------------------------------------------------- size-independent properties at BASELINE sizes
def test_full_c2_properties(cov, orc, engine):
    """1 M candidates x 5 UAVs on the 256 x 256 fire grid: (1) the objective is invariant under a
    permutation of the UAVs' discs except for the order-dependent penalty sum, whose terms we
    permute consistently so it is identical too when r_max is uniform and the sum is exact...
    we compare counts; (2) obj == -w*count + 1e5*violation recomputed in NumPy; (3) the span and
    brute kernels agree on the whole batch; (4) a 2000-candidate sample equals the oracle."""
    n = 256
    d = 500.0 / n
    bits, _ = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    engine.set_grid_bits(bits, n, n, d, d)
    N, B = 5, 1_000_000
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max)
    X = cov.synth.random_candidates(B, N, seed=1)
    a = engine.eval_batch(X)
    ll = engine.last_launch()
    # (the last launch of a host-path call is its short tail slice: at most one persistent CTA per SM)
    assert ll["kernel"] == cov.KERNEL_SPAN and ll["planes_in_smem"] == 1 and 1 <= ll["grid"] <= 148
    perm = np.array([3, 0, 4, 1, 2])
    Xp = np.concatenate([X[:, perm], X[:, N + perm], X[:, 2 * N + perm]], axis=1)
    b = engine.eval_batch(Xp)
    assert np.array_equal(a["count"], b["count"])
    viol = np.zeros(B)
    for i in range(N):
        viol = viol + np.abs(X[:, 2 * N + i] - r_max[i])
    assert np.array_equal(a["obj"], -(d * d * a["count"].astype(np.float64)) + viol * 1e5)
    engine.set_option(cov.OPT_KERNEL, KERNELS["brute"])
    c = engine.eval_batch(X[:100_000])
    assert np.array_equal(c["count"], a["count"][:100_000]) and np.array_equal(c["obj"], a["obj"][:100_000])
    idx = np.random.default_rng(0).choice(B, 2000, replace=False)
    want = orc.eval_batch(X[idx], N, r_max, pts)
    assert np.array_equal(a["count"][idx], want["count"]) and np.array_equal(a["obj"][idx], want["obj"])


# ---------------------------------------------------------------- the callers: MADS and the receding horizon
def test_mads_on_gpu_objective_c1(cov, orc, kat):
    """Config 1: one MADS solve of FullSimulation.jl's default problem on the GPU objective."""
    CF, OPT, TC, ACC = cov.CellFunctions, cov.TDM_STATIC_opt, cov.TDM_Constraints, cov.AreaCoverageCalculation
    cells = CF.initialise_POI(CF.Cells(), "static")
    N, FOV = 5, 100 / 180 * math.pi
    r_max = np.full(N, 30.0 * T)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    cells = CF.rmvCoveredPOI(cells, x0)
    pts = cells.points_of_interest.data.copy()
    obj = OPT.createObjective(cells, N, r_max)
    cons3 = TC.create_cons3(ACC.make_circles(x0), FOV, 10 * np.ones(N))
    f0 = obj(x0)
    assert f0 == orc.objective(x0, r_max, pts)[0]
    res, runtime, st = cov.mads.optimize(x0, obj, [TC.cons1, cons3], [], 100, seed=5, return_stats=True)
    assert runtime > 0 and st["batches"] >= 2 and st["evaluations"] > 30
    assert np.all(res == np.rint(res))                       # granularity 1.0
    assert orc.cons3(res, x0, T, np.full(N, 10.0))           # extreme barrier held
    f1 = obj(res)
    assert f1 < f0 and f1 == orc.objective(res, r_max, pts)[0]
    cells.close()


def test_receding_horizon_fire_c5(cov, orc, fire_rows):
    """Config 5: 20 fire-growth steps, each re-optimised with MADS on the GPU objective; the cell list
    after every step equals the oracle's replay of the same UAV positions."""
    CF, FS = cov.CellFunctions, cov.FullSimulation
    params = FS.SimulationParameters(environment_type="dynamic", N_iter=30, seed=11)
    cells = CF.initialise_POI(CF.Cells(), "dynamic", fire_rows=fire_rows)
    N = params.N
    start = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 330.0)
    r_max = params.h_max * T * np.ones(N)
    inp, outp, runtimes, objs = FS.run_simulation(cells, start, cov.TDM_Constraints.cons1, [], N, r_max, params,
                                                  Nt_sim=20)
    assert len(outp) == 20 and all(r > 0 for r in runtimes)
    # replay on the oracle: same list evolution, same objective value at every step's result
    ref = np.concatenate(fire_rows[:10])
    pre = start
    for t in range(1, 21):
        if t != 1:
            ref = np.concatenate([ref, fire_rows[t + 10 - 1]])
        ref = orc.rmvCoveredPOI(pre, ref)
        assert orc.cons3(outp[t - 1], pre, T, np.full(N, 10.0))
        assert objs[t - 1] == orc.objective(outp[t - 1], r_max, ref)[0]
        pre = outp[t - 1]
    assert np.array_equal(cells.points_of_interest.data, ref)
    cells.close()


# ---------------------------------------------------------------- forest-fire automaton on the device
def test_fire_automaton_matches_oracle(cov, orc, engine):
    """DynamicArea.jl's update_grid on the device: grid state and the pushed list entries (with their
    duplicates) equal the C restatement fed with the same Philox uniforms, step by step; then the
    objective on the device-grown store equals the oracle on the replayed list."""
    ff = cov.DynamicArea.ForestFire(engine, seed=2026)
    nx, ny = ff.nx, ff.ny
    assert (nx, ny) == (100, 100)
    grid = ff.initial_grid.T.ravel().copy()
    ii, jj = np.nonzero(ff.initial_grid == 2)
    order = np.lexsort((ii, jj))  # DynamicArea.jl:38-42: y outer, x inner
    pts = np.stack([(ii[order] + 1) * 5.0 - 2.5, (jj[order] + 1) * 5.0 - 2.5, np.full(len(ii), 25.0),
                    np.full(len(ii), 25.0), np.zeros(len(ii))], axis=1)
    assert engine.grid_info()["n_entries"] == len(pts) == 21 * 3
    total_dups = 0
    for step in range(1, 41):
        pushed = ff.step()
        grid, new_pts = orc.fire_step(grid, nx, ny, 5.0, 5.0, 4.0, math.radians(270.0), 0.5, step, 2026)
        assert pushed == len(new_pts)
        pts = np.concatenate([pts, new_pts])
        assert np.array_equal(engine.fire_state(), grid)
        total_dups += len(new_pts) - len(np.unique(new_pts[:, :2], axis=0))
    assert total_dups > 0  # cells pushed more than once in a step, as in FirePoints.xlsx
    ref_mult = np.zeros(nx * ny, dtype=np.int64)
    np.add.at(ref_mult, cov.AreaCoverageCalculation.PointList(pts, nx, ny, 5.0, 5.0).cell_index(), 1)
    assert np.array_equal(engine.grid_cells(), ref_mult)
    N = 5
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max)
    rng = np.random.default_rng(12)
    X = rand_candidates(rng, 1000, N)
    X[:, N:2 * N] *= 0.8
    check_against_oracle(cov, orc, engine, X, N, r_max, pts)


# ---------------------------------------------------------------- continuous union-area variant
UNION_RTOL = 1e-9  # measured agreement of the FP64 kernel with the NumPy restatement; north_star allows 1e-5


def test_union_area_closed_forms_and_oracle(cov, npo, engine):
    lens = lambda d: 2 * math.pi - (2 * math.acos(d / 2) - d / 2 * math.sqrt(4 - d * d))  # noqa: E731  two unit discs
    cases = [
        ([0, 0, 1.0], math.pi),                                  # one disc
        ([0, 1, 0, 0, 1, 1.0], lens(1.0)),                        # lens
        ([0, 0.1, 0, 0, 2, 1.0], 4 * math.pi),                    # contained
        ([0, 0, 0, 0, 1, 1.0], math.pi),                          # identical
        ([0, 2, 0, 0, 1, 1.0], 2 * math.pi),                      # externally tangent
        ([0, 1, 0, 0, 2, 1.0], 4 * math.pi),                      # internally tangent
        ([0, 5, 0, 0, 1, 2.0], 5 * math.pi),                      # disjoint
        ([0, 1, 0, 0, 1, 0.0], math.pi),                          # a zero-radius disc
        ([3, 3, 3, 7, 7, 7, 2, 2, 2.0], 4 * math.pi),             # three identical
    ]
    for x, want in cases:
        n = len(x) // 3
        got = float(engine.union_area(np.array([x], dtype=np.float64), n)[0])
        assert abs(got - want) <= UNION_RTOL * max(want, 1.0), (x, got, want)
        assert abs(npo.union_area(x) - want) <= 1e-12 * max(want, 1.0)
        # the same case padded with zero-radius discs to 70 circles: the CTA-per-candidate kernel (N > 64)
        pad = 70 - n
        xp = np.concatenate([x[:n], np.zeros(pad), x[n:2 * n], np.zeros(pad), x[2 * n:], np.zeros(pad)])
        got = float(engine.union_area(xp[None, :], 70)[0])
        assert abs(got - want) <= UNION_RTOL * max(want, 1.0), ("padded", x, got, want)
    same = np.concatenate([np.full(100, 3.0), np.full(100, 7.0), np.full(100, 2.0)])
    assert abs(float(engine.union_area(same[None, :], 100)[0]) - 4 * math.pi) <= UNION_RTOL * 4 * math.pi  # 100 identical
    rng = np.random.default_rng(4)
    for n in (1, 2, 5, 20, 64, 65, 200):
        nb = 200 if n <= 64 else 40
        X = np.concatenate([rng.random((nb, 2 * n)) * 120, 2 + rng.random((nb, n)) * 30], axis=1)
        X[:20, :2 * n] = 50 + X[:20, :2 * n] * 0.05  # tight clusters: containment and many crossings
        got = engine.union_area(X, n)
        want = np.array([npo.union_area(x) for x in X])
        assert np.all(np.abs(got - want) <= UNION_RTOL * want), np.max(np.abs(got - want) / want)
        assert np.all(got <= np.sum(math.pi * X[:, 2 * n:] ** 2, axis=1) * (1 + 1e-12))
        assert np.all(got >= math.pi * np.max(X[:, 2 * n:], axis=1) ** 2 * (1 - 1e-12))
    assert cov.AreaCoverageCalculation.unionArea(np.array([0, 1, 0, 0, 1, 1.0]), engine) == pytest.approx(lens(1.0), rel=1e-12)
    with pytest.raises(cov.CoverageError):
        engine.union_area(np.zeros((1, 3 * 1025)), 1025)
    big = np.concatenate([rng.random((3, 2048)) * 500, 2 + rng.random((3, 1024)) * 20], axis=1)  # the library's maximum
    got = engine.union_area(big, 1024)
    want = np.array([npo.union_area(x) for x in big])
    assert np.all(np.abs(got - want) <= UNION_RTOL * want)


def test_union_area_vs_fine_grid_count(cov, orc, engine):
    """The discrete objective converges to the continuous one: on a fine dense grid, cell area x covered
    cells approaches the union area (inside the domain)."""
    n = 2048
    d = 500.0 / n
    engine.set_grid_full(n, n, d, d)
    N = 6
    engine.set_params(N, np.zeros(N), penalty_scale=0.0)
    rng = np.random.default_rng(8)
    X = np.concatenate([100 + rng.random((16, 2 * N)) * 300, 10 + rng.random((16, N)) * 25], axis=1)
    counts = engine.eval_batch(X)["count"]
    area = engine.union_area(X, N)
    assert np.all(np.abs(counts * d * d - area) <= 2e-3 * area)


def test_two_handles_from_two_threads(cov, orc):
    """Distinct handles used from distinct threads at the same time (DirectSearch's SetMaxEvals case)."""
    import threading
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    N = 5
    r_max = np.full(N, 30 * T)
    results, errors = {}, []

    def work(k):
        try:
            with cov.CoverageEngine(0) as e:
                e.set_grid_full(100, 100, 5.0, 5.0)
                e.set_params(N, r_max)
                X = cov.synth.random_candidates(3000, N, seed=100 + k)
                outs = [e.eval_batch(X)["obj"].copy() for _ in range(5)]
                ones = [e.eval_one(X[i]) for i in range(20)]
                results[k] = (X, outs, ones)
        except Exception as ex:  # noqa: BLE001
            errors.append(ex)

    threads = [threading.Thread(target=work, args=(k,)) for k in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    for k, (X, outs, ones) in results.items():
        want = orc.eval_batch(X, N, r_max, pts)["obj"]
        for o in outs:
            assert np.array_equal(o, want)
        assert ones == want[:20].tolist()


@pytest.mark.parametrize("dx,dy,nx,ny", [(0.7, 0.7, 200, 150), (1.3, 0.9, 96, 257), (5.0, 5.0, 100, 100),
                                          (500 / 256, 500 / 256, 256, 256), (1e-3, 1e-3, 64, 64), (1e4, 1e4, 40, 40)])
def test_span_vs_exact_kernel_stress(cov, engine, dx, dy, nx, ny):
    """Randomised stress: the FP32-certified span kernels against the FP64-per-cell exact kernel (itself
    checked against the oracle above) on lattices with non-representable pitches, tiny and huge scales,
    many candidates, several swarm sizes."""
    rng = np.random.default_rng(int(nx * 1000 + ny))
    fire = rng.random((nx, ny)) < 0.5
    engine.set_grid_bits(cov.synth.pack_bits(fire), nx, ny, dx, dy)
    ex, ey = nx * dx, ny * dy
    for N in (1, 3, 8, 13):
        B = 6000
        X = np.concatenate([rng.random((B, N)) * ex * 1.2 - 0.1 * ex, rng.random((B, N)) * ey * 1.2 - 0.1 * ey,
                            rng.random((B, N)) ** 2 * 0.3 * min(ex, ey)], axis=1)
        X[:500, :2 * N] = np.rint(X[:500, :2 * N] / dx) * dx          # centres on lattice lines
        X[:500, 2 * N:] = np.rint(X[:500, 2 * N:] / dx) * dx          # radii multiples of the pitch: ties
        engine.set_params(N, np.full(N, 0.1 * min(ex, ey)))
        engine.set_option(cov.OPT_KERNEL, KERNELS["exact"])
        want = engine.eval_batch(X)
        for kernel in ("span", "span_general"):
            engine.set_option(cov.OPT_KERNEL, KERNELS[kernel])
            got = engine.eval_batch(X)
            assert np.array_equal(got["count"], want["count"]), (kernel, N, np.flatnonzero(got["count"] != want["count"])[:5])
            assert np.array_equal(got["obj"], want["obj"])


def test_native_mads_solve(cov, orc):
    """cov_mads_solve: the whole solve inside the library.  Properties of the reference's settings (integer
    mesh, extreme barrier, no worse than the start) and the returned objective equals the oracle's value."""
    CF, OPT, TC, ACC = cov.CellFunctions, cov.TDM_STATIC_opt, cov.TDM_Constraints, cov.AreaCoverageCalculation
    cells = CF.initialise_POI(CF.Cells(), "static")
    N, FOV = 5, 100 / 180 * math.pi
    r_max = np.full(N, 30.0 * T)
    x0 = cov.Base_Functions.allocate_even_circles(15.0, N, 10 * T, 250.0, 250.0)
    cells = CF.rmvCoveredPOI(cells, x0)
    pts = cells.points_of_interest.data.copy()
    obj = OPT.createObjective(cells, N, r_max)
    cons3 = TC.create_cons3(ACC.make_circles(x0), FOV, 10 * np.ones(N))
    f0 = obj(x0)
    for seed in (1, 2, 3):
        res, runtime, st = OPT.optimize(x0, obj, [TC.cons1, cons3], [], 100, seed=seed, return_stats=True, native=True)
        assert st["batches"] >= 2 and st["evaluations"] > 30 and runtime > 0
        assert np.all(res == np.rint(res)) and orc.cons3(res, x0, T, np.full(N, 10.0))
        f1 = orc.objective(res, r_max, pts)[0]
        assert st["objective"] == f1 and f1 < f0
    # the Python driver and the native one start from the same point and both descend
    res_py, _, st_py = OPT.optimize(x0, obj, [TC.cons1, cons3], [], 100, seed=1, return_stats=True, native=False)
    assert st_py["objective"] < f0
    # a host-only constraint cannot be fused: native=None falls back to the Python driver, native=True refuses
    res2, _ = OPT.optimize(x0, obj, [TC.cons1, cons3, lambda x: True], [], 20, seed=1)
    assert np.all(res2 == np.rint(res2)) or np.array_equal(res2, x0)
    with pytest.raises(ValueError):
        OPT.optimize(x0, obj, [lambda x: True], [], 5, native=True)
    cells.close()


@pytest.mark.parametrize("N", [9, 33, 97, 1024])
def test_swarm_sizes_cta_kernel_vs_oracle(cov, orc, engine, fire_rows, N):
    """Swarm sizes just above the small-kernel limit, around the early/lazy fire-word switch (96), and at the
    library's maximum (1024), on the fire list with duplicates (multi-plane path) and on a dense grid."""
    rng = np.random.default_rng(N)
    allp = np.concatenate(fire_rows[:40])
    r_max = np.full(N, 30 * T)
    B = 24 if N < 1024 else 3
    X = np.concatenate([150 + rng.random((B, N)) * 250, 150 + rng.random((B, N)) * 220,
                        (5 + rng.random((B, N)) * 25) * T], axis=1)
    engine.set_points(allp, 100, 100, 5.0, 5.0)
    engine.set_params(N, r_max, sep_min=15.0)
    check_against_oracle(cov, orc, engine, X, N, r_max, allp, sep_min=15.0)
    assert engine.last_launch()["kernel"] == cov.KERNEL_SPAN_GENERAL
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    engine.set_grid_full(100, 100, 5.0, 5.0)
    engine.set_params(N, r_max, sep_min=15.0)
    check_against_oracle(cov, orc, engine, X, N, r_max, pts, sep_min=15.0)
    with pytest.raises(cov.CoverageError):
        engine.set_params(1025, np.zeros(1025))


def test_device_path_misaligned_and_odd_batches(cov, orc, engine):
    """cov_eval_batch_device with a candidate pointer that is only 8-byte aligned, batch sizes that are not
    multiples of the unit size, and every optional output switched off."""
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    engine.set_grid_full(100, 100, 5.0, 5.0)
    N = 5
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max)
    for B in (1, 31, 127, 129, 1001, 4097, 70001):
        X = cov.synth.random_candidates(B, N, seed=B)
        want = orc.eval_batch(X[:min(B, 1500)], N, r_max, pts)
        raw = engine.device_alloc(B * 3 * N * 8 + 16)
        d_obj = engine.device_alloc(B * 8)
        for shift in (0, 8):
            engine.memcpy_h2d(raw + shift, X)
            engine.eval_batch_device(raw + shift, B, d_obj)  # no count, no feasibility
            obj = np.empty(B)
            engine.memcpy_d2h(obj, d_obj)
            engine.sync()
            assert np.array_equal(obj[:len(want["obj"])], want["obj"]), (B, shift)
        only = engine.eval_batch(X, want_count=False, want_feasible=False)
        assert set(only) == {"obj"} and np.array_equal(only["obj"], obj)
        engine.device_free(raw)
        engine.device_free(d_obj)


def test_bench_line_contract(cov, tmp_path):
    """bench.py runs end to end on one GPU and prints ONE JSON line with the contract's keys; --dump-outputs writes
    the last timed launch's outputs."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dump = str(tmp_path / "dump")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "3", "--batch", "50000",
                        "--launches", "3", "--cpu-seconds", "0.5", "--dump-outputs", dump],
                       capture_output=True, text=True, timeout=280, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "roofline", "roofline_hbm", "cpu_baseline", "e2e", "e2e_pageable",
              "gpu_launches", "clocks", "extra_workloads", "h2d_ceiling_gbs", "h2d_ceiling_with_results_gbs"):
        assert k in d, k
    assert 0 < d["h2d_ceiling_with_results_gbs"] <= d["h2d_ceiling_gbs"] * 1.1
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["value"] > 0 and d["gpu_launches"] == 2 * 3
    # the bound that matters is instruction issue; a non-default batch may run an instantiation without a capture
    assert d["roofline"]["bound"] == "issue" and d["roofline"]["kernel"].startswith("span_small_kernel<")
    assert d["roofline"]["frac"] is None or 0 < d["roofline"]["frac"] < 1.0
    assert d["roofline_hbm"]["bound"] == "hbm" and 0 < d["roofline_hbm"]["frac"] < 1.0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["parity_on_sample"] is True
    assert d["e2e"]["h2d_bytes_per_step"] == 3 * 50000 * 120 and d["e2e"]["value"] > 0 and d["e2e_pageable"]["value"] > 0
    assert d["e2e_mesh"]["h2d_bytes_per_step"] == 3 * 50000 * 30 and d["e2e_mesh"]["value"] > 0
    assert d["e2e_mesh"]["parity_on_sample"] is True
    ex = {e["workload"][:2]: e for e in d["extra_workloads"]}
    assert set(ex) == {"C3", "C4", "C1"} and all(e["parity_on_sample"] is True for e in ex.values())
    # the named configs at their bench batch sizes MUST carry a live issue fraction from the committed capture
    for k in ("C3", "C4"):
        assert ex[k]["roofline"]["bound"] == "issue" and 0 < ex[k]["roofline"]["frac"] < 1.0, ex[k]["roofline"]
        assert ex[k]["kernel"].startswith("span_cta_kernel<") and ex[k]["value"] > 0
    assert ex["C1"]["poll_latency_us"] > 0 and ex["C1"]["mads_solve_ms"] > 0
    out = {f[:-4]: np.load(os.path.join(dump, f)) for f in os.listdir(dump)}
    assert set(out) == {"obj", "count", "feasible"} and all(len(a) == 50000 for a in out.values())
    assert out["obj"].dtype == np.float64 and out["count"].dtype == np.float64 and out["feasible"].dtype == np.float32
    assert out["count"].sum() == d["check"]["count_sum_last_launch"] and np.isfinite(out["obj"]).all()
    assert set(np.unique(out["feasible"])) <= {0.0, 1.0}


def test_reference_arm_does_not_load_the_product_library():
    """bench.py --impl reference times the CPU port only: libcoverage_cuda must not even be mapped."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0'];\n"
            "try:\n    runpy.run_path(sys.argv[0], run_name='__main__')\nexcept SystemExit:\n    pass\n"
            "maps = open('/proc/self/maps').read()\n"
            "print('MAPPED_PRODUCT', 'libcoverage_cuda' in maps, 'MAPPED_ORACLE', 'libcoverage_oracle' in maps)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=280, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "MAPPED_PRODUCT False MAPPED_ORACLE True" in r.stdout, r.stdout[-500:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["value"] > 0


@pytest.mark.parametrize("n,N,B", [(1024, 50, 100_000), (4096, 200, 4_000)])
def test_c3_c4_span_vs_brute_at_scale(cov, engine, n, N, B):
    """BASELINE's large shapes on many candidates: the CTA span kernel against the brute-force kernel (every
    cell of every non-empty fire word x every disc; itself checked against the oracle on small samples above).
    Candidates come from the device-side Philox generator, as BASELINE.md prescribes for C4."""
    d = 500.0 / n
    bits, _ = cov.synth.fire_grid(n)
    engine.set_grid_bits(bits, n, n, d, d)
    engine.set_params(N, np.full(N, 30 * T), sep_min=15.0)
    dX = engine.device_alloc(B * 3 * N * 8)
    outs = {}
    engine.generate_candidates(dX, B, N, seed=77)
    for name in ("span", "brute"):
        engine.set_option(cov.OPT_KERNEL, KERNELS[name])
        d_obj, d_cnt, d_fe = engine.device_alloc(B * 8), engine.device_alloc(B * 8), engine.device_alloc(B)
        engine.eval_batch_device(dX, B, d_obj, d_cnt, d_fe)
        obj, cnt, fe = np.empty(B), np.empty(B, dtype=np.int64), np.empty(B, dtype=np.uint8)
        engine.memcpy_d2h(obj, d_obj)
        engine.memcpy_d2h(cnt, d_cnt)
        engine.memcpy_d2h(fe, d_fe)
        engine.sync()
        outs[name] = (obj, cnt, fe)
        for p in (d_obj, d_cnt, d_fe):
            engine.device_free(p)
    engine.device_free(dX)
    assert np.array_equal(outs["span"][1], outs["brute"][1])
    assert np.array_equal(outs["span"][0], outs["brute"][0])
    assert np.array_equal(outs["span"][2], outs["brute"][2])
    assert outs["span"][1].min() > 0


@pytest.mark.parametrize("nx,ny", [(32, 4095), (96, 2048)])
def test_small_kernel_item_index_limits(cov, engine, nx, ny):
    """The small-swarm kernel packs the per-disc item prefixes of a candidate into 16-bit fields and finds
    the disc of an item with one packed compare.  Push the fields to their limits: 8 discs that each cover
    every row of the tallest grid the kernel takes (8 x 4095 = 32 760 items, just below 0x7fff), discs
    with no rows at all in between (equal prefixes), and mixtures; against the exact kernel."""
    rng = np.random.default_rng(nx + ny)
    fire = rng.random((nx, ny)) < 0.4
    dx = dy = 1.0
    engine.set_grid_bits(cov.synth.pack_bits(fire), nx, ny, dx, dy)
    N, B = 8, 600
    ex, ey = nx * dx, ny * dy
    X = np.empty((B, 3 * N))
    X[:, :N] = rng.random((B, N)) * ex
    X[:, N:2 * N] = rng.random((B, N)) * ey
    X[:, 2 * N:] = rng.random((B, N)) * 40.0
    X[:200, N:2 * N] = ey / 2 + rng.random((200, N))          # every disc covers every row ...
    X[:200, 2 * N:] = ey * (0.6 + rng.random((200, N)))       # ... of the grid: the largest item count
    far = rng.random((B, N)) < 0.3                            # discs with no row on the grid
    far[:100] = False
    X[:, N:2 * N][far] = -1e6
    X[300:330, 2 * N:] = 0.0                                  # all-empty candidates
    engine.set_params(N, np.full(N, 10.0))
    engine.set_option(cov.OPT_KERNEL, KERNELS["exact"])
    want = engine.eval_batch(X)
    assert engine.last_launch()["kernel"] == cov.KERNEL_EXACT
    engine.set_option(cov.OPT_KERNEL, KERNELS["span"])
    got = engine.eval_batch(X)
    assert engine.last_launch()["kernel"] == cov.KERNEL_SPAN       # the small-swarm kernel took it
    assert np.array_equal(got["count"], want["count"]), np.flatnonzero(got["count"] != want["count"])[:5]
    assert np.array_equal(got["obj"].view(np.uint64), want["obj"].view(np.uint64))
    assert want["count"][:100].min() == int(fire.sum())       # the full-cover candidates count every fire cell


def test_auto_routing_by_batch_size(cov, orc, engine):
    """COV_KERNEL_AUTO: poll-sized and mid-sized batches of a small swarm go to the CTA-per-candidate kernel
    (lower latency), large ones to the small-swarm kernel; the results do not depend on the route."""
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0)
    engine.set_grid_full(100, 100, 5.0, 5.0)
    N = 5
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max, sep_min=15.0)
    engine.set_option(cov.OPT_KERNEL, cov.KERNEL_AUTO)
    X = rand_candidates(np.random.default_rng(11), 6000, N)
    want = orc.eval_batch(X, N, r_max, pts, sep_min=15.0)
    for B, kernel in ((1, cov.KERNEL_SPAN_GENERAL), (30, cov.KERNEL_SPAN_GENERAL), (200, cov.KERNEL_SPAN_GENERAL),
                      (1000, cov.KERNEL_SPAN_GENERAL), (3000, cov.KERNEL_SPAN), (6000, cov.KERNEL_SPAN)):
        got = engine.eval_batch(X[:B])
        assert engine.last_launch()["kernel"] == kernel, (B, engine.last_launch())
        assert np.array_equal(got["count"], want["count"][:B]) and np.array_equal(got["feasible"], want["feasible"][:B])
        assert np.array_equal(got["obj"].view(np.uint64), want["obj"][:B].view(np.uint64))
    assert engine.eval_one(X[5]) == want["obj"][5]


# ---------------------------------------------------------------- round-2 regressions (ADVICE.md) and larger direct samples
def test_class_numbering_survives_removals(cov, orc, engine, fire_rows):
    """Two dyadic weight classes (25 and 250): after rmvCoveredPOI deletes the leading entries of the first
    class -- and then every entry of it -- the host list's order of first appearance no longer matches the
    device's class numbering; calculateArea must still pair counts with the right weights."""
    ACC = cov.AreaCoverageCalculation
    allp = np.concatenate(fire_rows[:30]).copy()
    assert allp[0, 3] == 25.0
    first_xy = allp[0, :2].copy()
    heavy = (allp[:, 0] > first_xy[0] + 40)
    allp[heavy, 3] = 250.0
    assert 0 < heavy.sum() < len(allp)
    pl = ACC.PointList(allp, 100, 100, 5.0, 5.0)
    res = ACC.ResidentList(pl, engine=engine)
    eng = res.sync()
    assert eng.grid_info()["area_exact"] == 1 and eng.class_weights() == [25.0, 250.0]
    rng = np.random.default_rng(5)
    probe = rand_candidates(rng, 40, 4)
    probe[:, 4:8] = 200 + probe[:, 4:8] * 0.3

    def check():
        for x in probe:
            area, cnt, _ = orc.calculateArea(x, res.points.data)
            assert ACC.calculateArea(x, res) == area
    check()
    # delete the leading entries of the light class: the host list now starts with ... whatever is left
    ACC.rmvCoveredPOI(np.array([first_xy[0], first_xy[1], 12.0]), res)
    assert np.array_equal(res.points.data, orc.rmvCoveredPOI(np.array([first_xy[0], first_xy[1], 12.0]), allp))
    check()
    # delete EVERY light entry (x <= first_x + 40): the host list has one distinct weight, the device still two classes
    light = res.points.data[res.points.data[:, 3] == 25.0]
    big = np.array([light[:, 0].min() - 200.0, light[:, 1].mean(), 0.0])
    big[2] = np.abs(light[:, 0] - big[0]).max() + 1.0
    while (res.points.data[:, 3] == 25.0).any():
        xy = res.points.data[res.points.data[:, 3] == 25.0][0, :2]
        ACC.rmvCoveredPOI(np.array([xy[0] - 30.0, xy[1], 32.0]), res)
    assert len(res.points) > 0 and (res.points.data[:, 3] == 250.0).all()
    check()


def test_store_state_after_relattice_and_failed_appends(cov, orc, engine):
    """ADVICE: (1) a grid setter after cov_fire_init must invalidate the automaton (its buffers belong to the old
    lattice); (2) a failing append leaves store, planes and counts exactly as they were."""
    rng = np.random.default_rng(12)
    state = (rng.random(40 * 40) < 0.7).astype(np.uint8)
    state[:80] = 2
    engine.fire_init(state, 40, 40, 5.0, 5.0)
    engine.fire_step(4.0, 270 / 180 * math.pi, 0.5, seed=3, step=1)
    engine.set_grid_full(300, 300, 1.0, 1.0)  # a LARGER lattice
    with pytest.raises(cov.CoverageError) as ei:
        engine.fire_step(4.0, 270 / 180 * math.pi, 0.5, seed=3, step=2)
    assert ei.value.code == cov._lib.COV_ERR_STATE
    with pytest.raises(cov.CoverageError):
        engine.fire_state()
    # mixed weights on one cell / multiplicity overflow: rejected, and nothing changed
    pts = orc.createPOI(5.0, 5.0, 20.0, 20.0)
    engine.set_points(pts, 20, 20, 5.0, 5.0)
    N = 2
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max)
    X = rand_candidates(rng, 300, N, extent=100.0)
    before = engine.eval_batch(X)
    info0, cells0 = engine.grid_info(), engine.grid_cells()
    bad = pts[:50].copy()
    bad[25:, 3] = 99.0
    with pytest.raises(cov.CoverageError):
        engine.add_points(bad)
    many = np.repeat(pts[7:8], 300, axis=0)  # 1 + 300 entries on one cell
    with pytest.raises(cov.CoverageError) as ei:
        engine.add_points(np.concatenate([pts[100:140], many]))
    assert ei.value.code == cov._lib.COV_ERR_LIMIT
    assert engine.grid_info() == info0 and np.array_equal(engine.grid_cells(), cells0)
    after = engine.eval_batch(X)
    assert np.array_equal(before["count"], after["count"]) and np.array_equal(before["obj"], after["obj"])
    engine.add_points(pts[:50])  # and a good append still works
    now = np.concatenate([pts, pts[:50]])
    check_against_oracle(cov, orc, engine, X, N, r_max, now)


def test_two_objectives_share_one_engine(cov, orc):
    """ADVICE: two closures on the same Cells with different r_max / fused constraints, called alternately."""
    CF, OPT, TC = cov.CellFunctions, cov.TDM_STATIC_opt, cov.TDM_Constraints
    cells = CF.initialise_POI(CF.Cells(), "static")
    pts = cells.points_of_interest.data
    N = 5
    r1, r2 = np.full(N, 30 * T), np.full(N, 12 * T)
    f1, f2 = OPT.createObjective(cells, N, r1), OPT.createObjective(cells, N, r2)
    rng = np.random.default_rng(2)
    X = rand_candidates(rng, 64, N)
    pre = X[0]
    f2.fuse([TC.create_cons3(pre, 100 / 180 * math.pi, 10.0)])
    for k in range(6):
        x = X[k]
        assert f1(x) == orc.objective(x, r1, pts)[0]
        assert f2(x) == orc.objective(x, r2, pts)[0]
        two = np.array([x[0], x[1], x[N], x[N + 1], x[2 * N], x[2 * N + 1]])  # calculateArea with another N in between
        assert cov.AreaCoverageCalculation.calculateArea(two, cells.resident()) == orc.calculateArea(two, pts)[0]
    o1 = f1.batch(X)
    o2, fe2 = f2.batch(X, want_feasible=True)
    o1b, fe1 = f1.batch(X, want_feasible=True)
    assert np.array_equal(o1, orc.eval_batch(X, N, r1, pts)["obj"]) and np.array_equal(o1, o1b) and fe1.all()
    want2 = orc.eval_batch(X, N, r2, pts, pre=pre, d_lim=10.0, tan_half_fov=T)
    assert np.array_equal(o2, want2["obj"]) and np.array_equal(fe2, want2["feasible"].astype(bool))
    # mesh indices through the same closure: an int16 matrix travels packed, same values as the Float64 one
    Q = cov.synth.mesh_candidates(64, N, seed=4)
    assert np.array_equal(f1.batch(Q), orc.eval_batch(Q.astype(np.float64), N, r1, pts)["obj"])
    assert np.array_equal(f1.batch(Q, granularity=0.5), f1.batch(Q.astype(np.float64) * 0.5))
    cells.close()


def _philox_batch(cov, engine, B, N, seed, first=0):
    dX = engine.device_alloc(B * 3 * N * 8)
    engine.generate_candidates(dX, B, N, seed=seed, first_index=first)
    X = np.empty((B, 3 * N))
    engine.memcpy_d2h(X, dX)
    engine.sync()
    engine.device_free(dX)
    return X


@pytest.mark.slow
def test_c3_direct_oracle_sample_10k(cov, orc, engine):
    """BASELINE.md section 3: C3 (50 UAVs, 1024^2, cons8) against the literal CPU restatement on >= 10^4
    candidates -- half NumPy-seeded, half generated on the device by Philox (what the full-size runs use)."""
    n, N = 1024, 50
    d = 500.0 / n
    bits, nset = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    engine.set_grid_bits(bits, n, n, d, d)
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max, sep_min=15.0)
    Xd = _philox_batch(cov, engine, 6000, N, seed=404, first=3_999_000)
    assert np.array_equal(Xd, cov.synth.philox_candidates(6000, N, 404, 3_999_000))
    X = np.concatenate([cov.synth.random_candidates(6000, N, seed=12), Xd])
    got = check_against_oracle(cov, orc, engine, X, N, r_max, pts, sep_min=15.0)
    assert len(X) >= 10_000 and got["count"].min() > 0


@pytest.mark.slow
def test_c4_direct_oracle_sample_1k(cov, orc, engine):
    """C4 (200 UAVs, 4096^2, cons8): >= 10^3 candidates against the literal CPU restatement (~10^12 predicate
    evaluations on the host cores), half of them Philox candidates from the far end of the 16 M index range."""
    n, N = 4096, 200
    d = 500.0 / n
    bits, nset = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    engine.set_grid_bits(bits, n, n, d, d)
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max, sep_min=15.0)
    Xd = _philox_batch(cov, engine, 512, N, seed=8, first=16_000_000 - 512)
    X = np.concatenate([cov.synth.random_candidates(512, N, seed=13), Xd])
    check_against_oracle(cov, orc, engine, X, N, r_max, pts, sep_min=15.0)
    assert len(X) >= 1000


def test_eval_batch_best_and_pipelined_argmin(cov, orc, engine):
    """cov_eval_batch_best = cov_eval_batch + the poll winner reduced on the device (what one rank contributes to the
    (min, index) exchange of a sharded poll); cov_argmin takes the sliced pipeline from 4 MiB of candidates on."""
    engine.set_grid_full(100, 100, 5.0, 5.0)
    N = 5
    r_max = np.full(N, 30 * T)
    rng = np.random.default_rng(78)
    pre = rand_candidates(rng, 1, N)[0]
    B = 150_000  # 18 MB of candidates: several 16 MiB-slices of the host pipeline
    X = pre + rng.normal(0, 3.5, (B, 3 * N))
    engine.set_params(N, r_max, prev_xyR=pre, d_lim=10.0, tan_half_fov=T)
    ref = engine.eval_batch(X)
    feas = ref["feasible"].astype(bool)
    assert 0 < feas.sum() < B
    masked = np.where(feas, ref["obj"], np.inf)
    for barrier in (True, False):
        r = engine.eval_batch_best(X, barrier=barrier)
        assert np.array_equal(r["obj"], ref["obj"]) and np.array_equal(r["count"], ref["count"])
        assert np.array_equal(r["feasible"], ref["feasible"])
        v = masked if barrier else ref["obj"]
        assert r["best"] == (v.min(), int(np.argmin(v)))
        assert engine.argmin(X, barrier=barrier) == r["best"]
    small = engine.eval_batch_best(X[:30])  # a poll set
    assert small["best"] == (masked[:30].min(), int(np.argmin(masked[:30]))) or not feas[:30].any()
    engine.set_params(N, r_max, prev_xyR=pre + 1000.0, d_lim=10.0, tan_half_fov=T)
    assert engine.eval_batch_best(X)["best"] == (math.inf, -1)
    # pinned buffers take the same route
    Xp = engine.pinned((B, 3 * N))
    Xp[:] = X
    engine.set_params(N, r_max, prev_xyR=pre, d_lim=10.0, tan_half_fov=T)
    out = {"obj": engine.pinned((B,)), "count": engine.pinned((B,), np.int64), "feasible": engine.pinned((B,), np.uint8)}
    r = engine.eval_batch_best(Xp, out=out)
    assert np.array_equal(out["obj"], ref["obj"]) and r["best"] == (masked.min(), int(np.argmin(masked)))


@pytest.mark.parametrize("dtype,g", [(np.int16, 1.0), (np.int16, 0.5), (np.int32, 0.1), (np.float32, 1.0)])
def test_packed_candidates_match_the_widened_matrix(cov, orc, engine, dtype, g):
    """cov_eval_batch_packed: mesh indices (int16 / int32, value = q * granularity) or float32 values, widened on the
    device -- results bit for bit those of cov_eval_batch on the Float64 matrix (and of the oracle on it), on every
    route: poll set (host-widened), sliced pipeline from pageable and from pinned memory, odd slice sizes, the winner."""
    n = 256
    d = 500.0 / n
    bits, _ = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    engine.set_grid_bits(bits, n, n, d, d)
    N, B = 5, 150_001  # odd on purpose: the last slice is ragged, the element count is not a multiple of 4
    r_max = np.full(N, 30 * T)
    if dtype is np.float32:
        Q = cov.synth.random_candidates(B, N, seed=31).astype(np.float32)
        X = Q.astype(np.float64)
    else:
        Q = cov.synth.mesh_candidates(B, N, seed=31, granularity=g, dtype=dtype)
        X = Q.astype(np.float64) * g
    pre = X[0].copy()
    engine.set_params(N, r_max, prev_xyR=pre, d_lim=200.0, tan_half_fov=T)
    ref = engine.eval_batch(X)
    assert 0 < ref["feasible"].sum() < B
    want = orc.eval_batch(X[:600], N, r_max, pts, pre=pre, d_lim=np.full(N, 200.0), tan_half_fov=T)
    for k in ("count", "feasible"):
        assert np.array_equal(ref[k][:600], want[k])
    assert same_doubles(ref["obj"][:600], want["obj"])

    def check(r, nb=B):
        assert same_doubles(r["obj"], ref["obj"][:nb])
        assert np.array_equal(r["count"], ref["count"][:nb]) and np.array_equal(r["feasible"], ref["feasible"][:nb])

    check(engine.eval_batch_packed(Q, g))                      # pageable, sliced pipeline
    for nb in (1, 30, 2184):                                   # poll sets
        check(engine.eval_batch_packed(Q[:nb], g), nb)
    check(engine.eval_batch_packed(Q[:40_003], g), 40_003)     # one ragged slice (the mid-size route of the doubles)
    masked = np.where(ref["feasible"].astype(bool), ref["obj"], np.inf)
    r = engine.eval_batch_packed(Q, g, best=True)
    check(r)
    assert r["best"] == (masked.min(), int(np.argmin(masked)))
    r = engine.eval_batch_packed(Q, g, best=True, barrier=False)
    assert r["best"] == (ref["obj"].min(), int(np.argmin(ref["obj"])))
    Qp = engine.pinned((B, 3 * N), dtype)                      # pinned: DMA'd in place, zero-copy results
    Qp[:] = Q
    out = {"obj": engine.pinned((B,)), "count": engine.pinned((B,), np.int64), "feasible": engine.pinned((B,), np.uint8)}
    check(engine.eval_batch_packed(Qp, g, out=out))
    for chunk in (999, 4097):                                  # odd slices: misaligned device slices (scalar widening)
        engine.set_option(cov.OPT_CHUNK, chunk)
        check(engine.eval_batch_packed(Q[:20_001], g), 20_001)
    engine.set_option(cov.OPT_CHUNK, 0)
    engine.set_option(cov.OPT_ZEROCOPY_OUT, 0)
    check(engine.eval_batch_packed(Qp, g, out=out))
    engine.set_option(cov.OPT_ZEROCOPY_OUT, 1)
    if dtype is np.int16 and g == 1.0:                         # several full slices (both raw slots reused)
        Bb = 700_001
        Qb = cov.synth.mesh_candidates(Bb, N, seed=32, dtype=dtype)
        big = engine.eval_batch(Qb.astype(np.float64))
        r = engine.eval_batch_packed(Qb, g, best=True)
        for k in ("obj", "count", "feasible"):
            assert np.array_equal(r[k], big[k]), k
        mb = np.where(big["feasible"].astype(bool), big["obj"], np.inf)
        assert r["best"] == (mb.min(), int(np.argmin(mb))) or not np.isfinite(mb.min())


def test_packed_candidates_large_swarm_and_errors(cov, orc, engine):
    """The CTA-per-candidate kernel behind the packed entry (50 UAVs, cons8), and the argument checks."""
    n = 256
    d = 500.0 / n
    bits, _ = cov.synth.fire_grid(n)
    pts = cov.synth.points_from_bits(bits, n, d, d)
    engine.set_grid_bits(bits, n, n, d, d)
    N, B = 50, 6_000
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max, sep_min=15.0)
    Q = cov.synth.mesh_candidates(B, N, seed=7)
    X = Q.astype(np.float64)
    r = engine.eval_batch_packed(Q, 1.0)
    want = orc.eval_batch(X[:200], N, r_max, pts, sep_min=15.0)
    assert np.array_equal(r["count"][:200], want["count"]) and same_doubles(r["obj"][:200], want["obj"])
    assert np.array_equal(r["feasible"][:200], want["feasible"])
    ref = engine.eval_batch(X)
    assert same_doubles(r["obj"], ref["obj"]) and np.array_equal(r["count"], ref["count"])
    import ctypes as C
    lib, h = cov._lib.lib, engine.handle
    obj = np.empty(4)
    bo, bi = C.c_double(), C.c_int64()
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    assert lib.cov_eval_batch_packed(h, p(Q), 9, 1.0, 4, p(obj), None, None, 1, None, None) == cov._lib.COV_ERR_INVALID
    assert lib.cov_eval_batch_packed(h, p(Q), 3, 0.0, 4, p(obj), None, None, 1, None, None) == cov._lib.COV_ERR_INVALID
    assert lib.cov_eval_batch_packed(h, p(Q), 3, math.nan, 4, p(obj), None, None, 1, None, None) == cov._lib.COV_ERR_INVALID
    assert lib.cov_eval_batch_packed(h, p(Q), 3, 1.0, 4, p(obj), None, None, 1, C.byref(bo), None) == cov._lib.COV_ERR_INVALID
    assert lib.cov_eval_batch_packed(h, None, 3, 1.0, 4, p(obj), None, None, 1, None, None) == cov._lib.COV_ERR_INVALID
    assert lib.cov_eval_batch_packed(h, p(Q), 3, 1.0, 4, None, None, None, 1, None, None) == cov._lib.COV_ERR_INVALID
    assert lib.cov_eval_batch_packed(h, p(Q), 3, 1.0, 0, p(obj), None, None, 1, None, None) == cov._lib.COV_OK
    assert lib.cov_eval_batch_packed(h, p(Q), 3, 1.0, 4, None, None, None, 1, C.byref(bo), C.byref(bi)) == cov._lib.COV_OK
    assert bi.value == int(np.argmin(np.where(ref["feasible"][:4].astype(bool), ref["obj"][:4], np.inf))) or bi.value == -1
