"""The host routes of the evaluation entry points.

Every route of cov_eval_batch / _ex / _packed (the small path with and without zero-copy, the mid-size zero-copy
launch, the sliced pipeline with pageable or pinned input) must return the same bytes for every set of result
columns, pinned, pageable or mixed, with the launches of the route it is meant to take, and the oracle's values.
Every poll-winner entry point must pick the lowest objective, a tie going to the earlier index.
"""
import ctypes as C
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

T = math.tan((100 / 180 * math.pi) / 2)
N = 5
B_MID = 200_003      # above the small path, below COV_ZC_MID_LIMIT; two default slices of the pipeline
CHUNK = 999          # COV_OPT_CHUNK of the sliced runs: several slices
ROW = 3 * N * 8
COLS = {"obj": ((), np.float64), "count": ((), np.int64), "class_count": ((2,), np.int64),
        "progressive": ((), np.float64), "feasible": ((), np.uint8)}
ALL = tuple(COLS)
MIXED_PINNED = ("obj", "class_count", "feasible")   # count and progressive stay pageable


def _two_class_store(engine, orc):
    """createPOI(5, 5, 100, 100) with a block of weight-100 entries: class_count has two columns."""
    pts = orc.createPOI(5.0, 5.0, 100.0, 100.0).copy()
    heavy = (pts[:, 0] > 150) & (pts[:, 0] < 350) & (pts[:, 1] > 200)
    pts[heavy, 3] = 100.0
    engine.set_points(pts, 100, 100, 5.0, 5.0)
    r_max = np.full(N, 30 * T)
    engine.set_params(N, r_max, sep_min=15.0)
    assert engine.grid_info()["n_classes"] == 2
    return pts, r_max


def _slices(B, chunk):
    return -(-B // chunk)


def _default_chunk(packed):
    slice_bytes = (32 << 20) if packed else (16 << 20)
    return max(1024, (slice_bytes // ROW) // 32 * 32)


def _outputs(engine, B, names, pinned):
    out = {}
    for k in names:
        shape, dt = COLS[k]
        a = engine.pinned((B,) + shape, dt) if k in pinned else np.empty((B,) + shape, dt)
        a.view(np.uint8)[...] = 0xA5    # whatever a route leaves unwritten shows
        out[k] = a
    return out


def _eval(engine, X, names, pinned=()):
    out = _outputs(engine, X.shape[0], names, pinned)
    before = engine.launch_count()
    r = engine.eval_batch(X, want_count="count" in names, want_feasible="feasible" in names,
                          want_class_count="class_count" in names, want_progressive="progressive" in names, out=out)
    return r, engine.launch_count() - before


def _packed(engine, Q, names, pinned=(), best=False):
    out = _outputs(engine, Q.shape[0], names, pinned)
    before = engine.launch_count()
    r = engine.eval_batch_packed(Q, 1.0, want_count="count" in names, want_feasible="feasible" in names, best=best,
                                 out=out)
    return r, engine.launch_count() - before


def _same(r, ref, names, what):
    for k in names:
        assert r[k].tobytes() == ref[k][:r[k].shape[0]].tobytes(), (what, k)


def test_column_matrix(cov, orc, engine):
    pts, r_max = _two_class_store(engine, orc)
    Q = cov.synth.mesh_candidates(B_MID, N, seed=11)          # on the mesh: the packed entry sees the same doubles
    X = Q.astype(np.float64)
    Xp = engine.pinned(X.shape)
    Xp[:] = X
    Qp = engine.pinned(Q.shape, np.int16)
    Qp[:] = Q
    colsets = [("obj",), ALL]

    # the sliced pipeline: pageable / pinned input, zero-copy on / off, every column set
    engine.set_option(cov.OPT_CHUNK, CHUNK)
    ref, n = _eval(engine, X, ALL)
    assert n == _slices(B_MID, CHUNK)
    for zc in (1, 0):
        engine.set_option(cov.OPT_ZEROCOPY_OUT, zc)
        for Xin in (X, Xp):
            for names, pinned in [(c, ()) for c in colsets] + [(c, c) for c in colsets] + [(ALL, MIXED_PINNED)]:
                r, n = _eval(engine, Xin, names, pinned)
                _same(r, ref, names, ("sliced", zc, Xin is Xp, pinned))
                assert n == _slices(B_MID, CHUNK), ("sliced", zc, names, pinned)
        for Qin in (Q, Qp):                                   # plus one widening launch per slice
            r, n = _packed(engine, Qin, ("obj", "count", "feasible"), ("obj",))
            _same(r, ref, ("obj", "count", "feasible"), ("packed sliced", zc))
            assert n == 2 * _slices(B_MID, CHUNK)
    engine.set_option(cov.OPT_CHUNK, 0)

    # the small path: the pinned poll scratch, with and without zero-copy; a packed poll set is widened on the host
    for zc in (1, 0):
        engine.set_option(cov.OPT_ZEROCOPY_OUT, zc)
        for B in (1, 30, 2184):
            for names, pinned in [(c, ()) for c in colsets] + [(ALL, MIXED_PINNED)]:
                r, n = _eval(engine, X[:B], names, pinned)
                _same(r, ref, names, ("small", zc, B, pinned))
                assert n == 1, ("small", zc, B, names)
            r, n = _packed(engine, Q[:B], ("obj", "count", "feasible"))
            _same(r, ref, ("obj", "count", "feasible"), ("packed small", zc, B))
            assert n == 1

    # mid-size: pinned input and outputs, one zero-copy launch; a pageable column sends the call to the pipeline
    engine.set_option(cov.OPT_ZEROCOPY_OUT, 1)
    for names in colsets:
        r, n = _eval(engine, Xp, names, names)
        _same(r, ref, names, ("mid", names))
        assert n == 1
    r, n = _eval(engine, Xp, ALL, MIXED_PINNED)
    _same(r, ref, ALL, "default slices, mixed")
    assert n == _slices(B_MID, _default_chunk(False)) == 2
    r, n = _packed(engine, Q, ("obj", "count", "feasible"))
    _same(r, ref, ("obj", "count", "feasible"), "packed default slices")
    assert n == 2 * _slices(B_MID, _default_chunk(True))

    # the oracle on a sample: count, feasibility, objective bits, per-class counts
    assert 0 < int(ref["feasible"].sum()) < B_MID
    idx = np.concatenate([np.arange(64), np.random.default_rng(3).choice(np.arange(64, B_MID), 64, replace=False)])
    want = orc.eval_batch(X[idx], N, r_max, pts, sep_min=15.0)
    assert np.array_equal(ref["count"][idx], want["count"])
    assert np.array_equal(ref["feasible"][idx], want["feasible"])
    assert ref["obj"][idx].tobytes() == want["obj"].tobytes()
    weights = engine.class_weights()
    class_of = np.array([weights.index(w) for w in pts[:, 3]], dtype=np.int32)
    for i in idx[:48]:
        assert np.array_equal(ref["class_count"][i], orc.class_counts(X[i], pts, class_of, 2)), i


# ---------------------------------------------------------------------------------------------- the poll winner
def _winner(obj, feasible, barrier):
    ok = ~np.isnan(obj) & (feasible.astype(bool) if barrier else True)
    if not ok.any():
        return math.inf, -1
    v = obj[ok].min()
    return float(v), int(np.flatnonzero(ok & (obj == v))[0])


def _planted(pool_obj, pool_ok, B, at, rng):
    """Row indices into the pool: the pool's unique best candidate at the indices `at`, other rows elsewhere."""
    v = pool_obj[pool_ok].min()
    best = int(np.flatnonzero(pool_ok & (pool_obj == v))[0])
    others = np.flatnonzero(pool_obj != v)
    rows = rng.choice(others, B)
    rows[list(at)] = best
    return rows


def _plants(B):
    return [[0], [1, 2], [B // 2, B // 2 + 1, B - 1], [B - 1], [7, B - 1]]


def test_winner_grid_entries(cov, orc, engine):
    _two_class_store(engine, orc)
    pool_q = cov.synth.mesh_candidates(256, N, seed=21)
    pool = pool_q.astype(np.float64)
    p = engine.eval_batch(pool)
    rng = np.random.default_rng(5)
    for B in (3000, B_MID):                                   # cov_argmin below and above its 4 MiB switch
        for barrier in (True, False):
            ok = p["feasible"].astype(bool) if barrier else np.ones(len(pool), bool)
            for at in _plants(B):
                rows = _planted(p["obj"], ok, B, at, rng)
                X, Q = pool[rows], pool_q[rows]
                per = engine.eval_batch(X)
                want = _winner(per["obj"], per["feasible"], barrier)
                assert want[1] == at[0]
                assert engine.eval_batch_best(X, barrier=barrier)["best"] == want, (B, barrier, at)
                assert engine.eval_batch_packed(Q, 1.0, best=True, barrier=barrier)["best"] == want
                assert engine.argmin(X, barrier=barrier) == want, (B, barrier, at)
    # every candidate infeasible: (inf, -1) with the barrier, the raw minimum without
    x = pool[0].copy()
    x[1:N] = x[0]
    x[N + 1:2 * N] = x[N]                                      # every disc at one point: cons8 fails
    X = np.repeat(x[None, :], 3000, axis=0)
    per = engine.eval_batch(X)
    assert not per["feasible"].any()
    assert engine.eval_batch_best(X, barrier=True)["best"] == (math.inf, -1)
    assert engine.argmin(X, barrier=True) == (math.inf, -1)
    assert engine.eval_batch_packed(X.astype(np.int16), 1.0, best=True, barrier=True)["best"] == (math.inf, -1)
    assert engine.argmin(X, barrier=False) == (per["obj"][0], 0)
    assert engine.eval_batch_best(X, barrier=False)["best"] == (per["obj"][0], 0)
    # no candidates
    E = np.empty((0, 3 * N))
    assert engine.eval_batch_best(E)["best"] == (math.inf, -1)
    assert engine.argmin(E) == (math.inf, -1)
    assert engine.eval_batch_packed(E.astype(np.int16), 1.0, best=True)["best"] == (math.inf, -1)


def test_winner_region(cov, engine):
    engine.set_region(0.0, 0.0, 500.0, 500.0, covered=np.array([[250.0, 250.0, 40.0], [100.0, 400.0, 25.0]]))
    engine.set_params(N, np.full(N, 30 * T), sep_min=15.0)
    pool = cov.synth.mesh_candidates(256, N, seed=22).astype(np.float64)
    p = engine.eval_region_batch(pool)
    rng = np.random.default_rng(6)
    for barrier in (True, False):
        ok = p["feasible"].astype(bool) if barrier else np.ones(len(pool), bool)
        for at in _plants(3000):
            X = pool[_planted(p["obj"], ok, 3000, at, rng)]
            r = engine.eval_region_batch(X, best=True, barrier=barrier)
            want = _winner(r["obj"], r["feasible"], barrier)
            assert want[1] == at[0] and r["best"] == want, (barrier, at)
    x = pool[0].copy()
    x[1:N] = x[0]
    x[N + 1:2 * N] = x[N]
    X = np.repeat(x[None, :], 100, axis=0)
    r = engine.eval_region_batch(X, best=True, barrier=True)
    assert not r["feasible"].any() and r["best"] == (math.inf, -1)
    assert engine.eval_region_batch(X, best=True, barrier=False)["best"] == (r["obj"][0], 0)
    assert engine.eval_region_batch(np.empty((0, 3 * N)), best=True)["best"] == (math.inf, -1)


def test_winner_multi(cov, orc):
    lib = cov._lib.lib
    devs = (C.c_int * 2)(0, 0)
    m = C.c_void_p()
    assert lib.cov_multi_create(devs, 2, C.byref(m)) == 0
    try:
        r_max = np.full(N, 30 * T)
        for k in range(2):
            h = lib.cov_multi_handle(m, k)
            assert lib.cov_set_grid_full(h, 100, 100, 5.0, 5.0) == 0
            assert lib.cov_set_params(h, N, r_max.ctypes.data, 1e5, None, None, T, 15.0, 0) == 0
        pool = cov.synth.mesh_candidates(256, N, seed=23).astype(np.float64)
        want_pool = orc.eval_batch(pool, N, r_max, orc.createPOI(5.0, 5.0, 100.0, 100.0), sep_min=15.0)
        rng = np.random.default_rng(7)

        def multi(X, barrier):
            bo, bi = C.c_double(), C.c_int64()
            assert lib.cov_multi_argmin(m, X.ctypes.data, X.shape[0], barrier, C.byref(bo), C.byref(bi)) == 0
            return bo.value, bi.value

        B = 3001                                               # shards 0..1500 and 1501..3000
        for barrier in (1, 0):
            ok = want_pool["feasible"].astype(bool) if barrier else np.ones(len(pool), bool)
            for at in _plants(B) + [[1501, 1502]]:
                rows = _planted(want_pool["obj"], ok, B, at, rng)
                X = np.ascontiguousarray(pool[rows])
                want = _winner(want_pool["obj"][rows], want_pool["feasible"][rows], barrier)
                assert want[1] == at[0] and multi(X, barrier) == want, (barrier, at)
        x = pool[0].copy()
        x[1:N] = x[0]
        x[N + 1:2 * N] = x[N]
        X = np.ascontiguousarray(np.repeat(x[None, :], 100, axis=0))
        assert multi(X, 1) == (math.inf, -1)
        assert multi(np.empty((0, 3 * N)), 1) == (math.inf, -1)
    finally:
        lib.cov_multi_destroy(m)
