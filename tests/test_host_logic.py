"""CPU-only: host-side logic around the path (data formats, synthetic inputs, list handling)."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_fire_rows_roundtrip(cov, fire_rows, tmp_path):
    p = str(tmp_path / "rows.npz")
    cov.fire_io.save_fire_rows_npz(p, fire_rows)
    back = cov.fire_io.load_fire_rows_npz(p)
    assert len(back) == len(fire_rows) and all(np.array_equal(a, b) for a, b in zip(back, fire_rows))


def test_fire_rows_on_lattice(cov, fire_rows):
    allp = np.concatenate(fire_rows)
    pl = cov.AreaCoverageCalculation.PointList(allp, 100, 100, 5.0, 5.0)
    idx = pl.cell_index()
    i, j = idx % 100 + 1, idx // 100 + 1
    assert np.array_equal(i * 5.0 - 2.5, allp[:, 0]) and np.array_equal(j * 5.0 - 2.5, allp[:, 1])
    assert allp[:, 0].min() == 7.5 and allp[:, 0].max() == 492.5 and allp[:, 1].max() == 352.5


def test_pack_unpack_bits(cov):
    rng = np.random.default_rng(1)
    for nx, ny in ((100, 100), (256, 64), (33, 7), (1, 1), (64, 3)):
        fire = rng.random((nx, ny)) < 0.4
        bits = cov.synth.pack_bits(fire)
        assert bits.shape == (ny, (nx + 31) // 32) and bits.dtype == np.uint32
        assert np.array_equal(cov.synth.unpack_bits(bits, nx), fire)
        i, j = nx // 2, ny // 2
        assert bool((bits[j, i >> 5] >> np.uint32(i & 31)) & np.uint32(1)) == bool(fire[i, j])


def test_fire_grid_deterministic(cov):
    a, na = cov.synth.fire_grid(256)
    b, nb = cov.synth.fire_grid(256)
    assert np.array_equal(a, b) and na == nb and 0.15 < na / 256 ** 2 < 0.5
    d, nd = cov.synth.fire_grid(64, dense=True)
    assert nd == 64 * 64


def test_points_from_bits_matches_createPOI(cov, orc):
    bits, n = cov.synth.fire_grid(32, dense=True)
    pts = cov.synth.points_from_bits(bits, 32, 5.0, 5.0)
    assert np.array_equal(pts, orc.createPOI(5.0, 5.0, 32.0, 32.0))
    assert np.array_equal(cov.AreaCoverageCalculation.createPOI(5.0, 5.0, 32.0, 32.0).data, pts)


def test_pointlist_infer(cov, fire_rows):
    pl = cov.AreaCoverageCalculation.PointList.infer(np.concatenate(fire_rows[:10]))
    assert (pl.dx, pl.dy) == (5.0, 5.0) and pl.nx >= 60 and pl.ny >= 69


def test_make_circles_roundtrip(cov):
    x = np.arange(15, dtype=np.float64)
    c = cov.AreaCoverageCalculation.make_circles(x)
    assert (c[1].x, c[1].y, c[1].R) == (1.0, 6.0, 11.0)
    assert np.array_equal(cov.AreaCoverageCalculation.make_MADS(c), x)


def test_allocate_even_circles(cov, kat):
    import math
    T = math.tan((100 / 180 * math.pi) / 2)
    x = cov.Base_Functions.allocate_even_circles(15.0, 5, 10 * T, 250.0, 250.0)
    assert x.tolist() == kat["kat3"]["x"]


def test_candidates_shapes(cov):
    X = cov.synth.random_candidates(100, 5, seed=1)
    assert X.shape == (100, 15) and X[:, :10].min() >= 0 and X[:, :10].max() < 500
    T = cov.TAN_HALF_FOV_DEFAULT
    assert X[:, 10:].min() >= 5 * T and X[:, 10:].max() <= 30 * T
    P = cov.synth.philox_candidates(64, 3, seed=99, first_index=1 << 33)
    assert P.shape == (64, 9) and len(np.unique(P)) == P.size
    assert np.array_equal(P[10:20], cov.synth.philox_candidates(10, 3, seed=99, first_index=(1 << 33) + 10))


def test_every_python_file_compiles():
    """tools/, the package, bench.py and __graft_entry__.py are syntactically valid (the GPU-side tools are not
    exercised by the CPU suite otherwise)."""
    import glob
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = glob.glob(os.path.join(root, "tools", "*.py")) + glob.glob(os.path.join(root, "oracle", "*.py")) + \
        glob.glob(os.path.join(root, "maximumareacoverageoptimization.jl_b200", "*.py")) + \
        [os.path.join(root, "bench.py"), os.path.join(root, "__graft_entry__.py"), os.path.join(root, "coverage_b200.py")]
    assert len(files) > 30
    for f in files:
        with open(f) as fh:
            compile(fh.read(), f, "exec")


def test_bench_issue_roofline_helpers(tmp_path, monkeypatch):
    """bench.py's live issue-slot roofline: the kernel key names the template instantiation, a missing capture fails
    loudly for the named workload, a capture from other sources is flagged stale."""
    import importlib.util
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    small = {"kernel": 1, "multi": 0, "chunk": 16, "max_warps": 20, "plane_mode": -1}
    cta = {"kernel": 4, "multi": 0, "chunk": 8, "max_warps": 0, "plane_mode": 4}
    assert bench.kernel_key(small) == "span_small_kernel<0,16,20>" and bench.kernel_key(cta) == "span_cta_kernel<0,4,8>"
    prof = {"source_sha": bench.source_sha(), "kernels": {"c2|span_small_kernel<0,16,20>": {
        "warp_instr_per_candidate": 600.0, "dram_bytes_per_launch": 1.27e8, "issue_active_pct": 74.0}}}
    v = bench.issue_view(prof, "c2", "span_small_kernel<0,16,20>", 1_000_000, 0.7, 1965.0, strict=True)
    assert v["bound"] == "issue" and abs(v["achieved"] - 600.0 * 1e6 / 0.7e-3) < 1 and "profile_stale" not in v
    assert abs(v["peak"] - 148 * 4 * 1965e6) < 1 and abs(v["frac"] - v["achieved"] / v["peak"]) < 1e-12
    prof["source_sha"] = "0" * 16
    assert bench.issue_view(prof, "c2", "span_small_kernel<0,16,20>", 1_000_000, 0.7, 1965.0, strict=True)["profile_stale"]
    monkeypatch.delenv("COV_BENCH_ALLOW_MISSING_PROFILE", raising=False)
    with pytest.raises(SystemExit):
        bench.issue_view(prof, "c2", "span_small_kernel<0,4,20>", 1_000_000, 0.7, 1965.0, strict=True)
    assert bench.issue_view(prof, "c2", "span_small_kernel<0,4,20>", 50_000, 0.1, 1965.0, strict=False)["frac"] is None
    # the committed capture covers the bench workloads
    with open(os.path.join(root, "profiles", "r2_issue.json")) as f:
        committed = json.load(f)
    assert {k.split("|")[0] for k in committed["kernels"]} >= {"c2", "c3", "c4"}
    assert len(bench.source_sha()) == 16 and bench.source_sha() == bench.source_sha()


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: obj / count as float64 and feasible as float32, one row per candidate; above 64 MB in
    all, the same seeded sample of rows on every run, with their row numbers in index.npy."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(3)

    def outputs(n):
        return {"obj": rng.normal(size=n), "count": rng.integers(0, 1 << 16, n),
                "feasible": rng.integers(0, 2, n).astype(np.uint8)}

    def load(d):
        return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}

    small = outputs(1000)
    bench.dump_outputs(str(tmp_path / "small"), small)
    got = load(tmp_path / "small")
    assert set(got) == {"obj", "count", "feasible"}
    assert got["obj"].dtype == np.float64 and got["count"].dtype == np.float64 and got["feasible"].dtype == np.float32
    for k in got:
        assert np.array_equal(got[k], small[k]), k

    n = bench.DUMP_LIMIT_BYTES // 20 + 12345  # 20 bytes per row once widened: just over the limit
    big = outputs(n)
    bench.dump_outputs(str(tmp_path / "a"), big)
    bench.dump_outputs(str(tmp_path / "b"), big)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert set(a) == {"obj", "count", "feasible", "index"} and all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(os.path.getsize(os.path.join(tmp_path, "a", f)) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_LIMIT_BYTES
    idx = a["index"].astype(np.int64)
    assert np.array_equal(idx.astype(np.float64), a["index"]) and np.all(np.diff(idx) > 0) and idx[-1] < n
    assert len(idx) > n // 2
    for k in ("obj", "count", "feasible"):
        assert np.array_equal(a[k], big[k][idx]), k


def test_pack_candidates_is_lossless_or_refuses(cov):
    """Mesh indices for cov_eval_batch_packed: what the device computes from them, (double)q * granularity, must be the
    caller's Float64 candidates bit for bit -- pack_candidates checks exactly that and refuses anything else."""
    import pytest
    from coverage_b200 import mads
    rng = np.random.default_rng(3)
    # trial points of the poll driver ARE on the mesh: _snap writes rint(v / g) * g, the same product the device forms
    for g in (1.0, 0.5, 0.25, 0.1, 2.0):
        P = mads._snap(rng.uniform(-50, 550, (400, 15)), np.full(15, g))
        for dt in (np.int16, np.int32):
            Q = cov.pack_candidates(P, g, dt)
            assert Q.dtype == dt and np.array_equal(Q.astype(np.float64) * g, P)  # (by value: rint gives -0.0 too)
    Q = cov.synth.mesh_candidates(1000, 5, seed=1)
    assert np.array_equal(cov.pack_candidates(Q.astype(np.float64)), Q)
    X = cov.synth.random_candidates(100, 5, seed=2)
    with pytest.raises(ValueError, match="not on the mesh"):
        cov.pack_candidates(X)                                   # random reals are not integers
    with pytest.raises(ValueError, match="not on the mesh"):
        cov.pack_candidates(X, dtype=np.float32)                 # nor FP32-representable
    F = X.astype(np.float32).astype(np.float64)
    assert np.array_equal(cov.pack_candidates(F, dtype=np.float32).astype(np.float64), F)
    with pytest.raises(ValueError, match="does not fit"):
        cov.pack_candidates(np.array([[40000.0, 1.0, 2.0]]))     # beyond int16
    assert cov.pack_candidates(np.array([[40000.0, 1.0, 2.0]]), dtype=np.int32).tolist() == [[40000, 1, 2]]
    with pytest.raises(ValueError):
        cov.pack_candidates(np.array([[np.nan, 1.0, 2.0]]))
    with pytest.raises(ValueError):
        cov.pack_candidates(np.ones((1, 3)), granularity=0.0)
    with pytest.raises(TypeError):
        cov.pack_candidates(np.ones((1, 3)), dtype=np.int64)
    # a granularity that is not a power of two: 0.1 * q is one rounded product on both sides, so values made that
    # way pack; the same numbers typed in decimal may not (0.3 != 3 * 0.1 in binary64)
    assert cov.pack_candidates(np.array([[3 * 0.1]]), 0.1).tolist() == [[3]]
    with pytest.raises(ValueError, match="not on the mesh"):
        cov.pack_candidates(np.array([[0.3]]), 0.1)
