"""Every compiled instantiation of the two span kernels, reached through the launchers and compared with the C oracle.

CPU: the instantiations nvcc built (cuobjdump) are exactly the rows of SMALL_VARIANTS and CTA_VARIANTS below, so a new
template argument without a test row fails on a machine without a GPU.

GPU: every row is driven to its instantiation through the public inputs only (store kind, N, batch size,
COV_OPT_WARPS_PER_CTA / CTAS_PER_SM / PLANE_MODE), cov_last_launch must name it, and count, feasibility, objective
bits, progressive bits and (multi-plane stores) the per-class counts must equal the oracle's on every row, with
COV_OPT_FORCE_EXACT 0 and 1.  Then the band and unit edges of the CTA kernel under forced band heights, and chords
wide enough for the whole-word paint loops."""
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

# span_small_kernel<MULTI, CHUNK, MAXW, FEW>.  FEW = N <= 5.  32-candidate units of 6 to 8 UAVs never get more than
# 20 warps (the shared memory of 21 is more than a CTA can have), so (*, 32, 24, 0) is not built.
SMALL_VARIANTS = [(m, c, w, f) for m in (0, 1) for c in (4, 8, 16, 32) for w in (20, 24) for f in (0, 1)
                  if not (c == 32 and w == 24 and f == 0)]
# span_cta_kernel<MULTI, PLANES, THREADS, CTAS>, with the options that reach each one (N = 72: more than 64 discs
# take 256-thread CTAs; a multi-plane store resolves every plane mode to 0)
CTA_REACH = {
    (0, 0, 256, 3): dict(N=5, mode=0),
    (0, 1, 128, 8): dict(N=5, mode=1),
    (0, 1, 256, 3): dict(N=72, mode=1),
    (0, 2, 256, 3): dict(N=5, mode=2),
    (0, 3, 256, 3): dict(N=5, mode=3),
    (0, 4, 128, 8): dict(N=5, mode=4),
    (0, 4, 256, 3): dict(N=5, mode=4, ctas=3),
    (0, 4, 256, 4): dict(N=5, mode=4, ctas=4),
    (1, 0, 128, 8): dict(N=5, mode=-1),
    (1, 0, 256, 3): dict(N=72, mode=2),
}
CTA_VARIANTS = sorted(CTA_REACH)


# ---------------------------------------------------------------- CPU: the inventory
@pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)), reason="needs cuobjdump and the built library")
def test_every_span_instantiation_has_a_row():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    names = set(re.findall(r"Function (\S+):", out))
    small, cta = set(), set()
    for n in names:
        m = re.search(r"span_small_kernelILb([01])ELi(\d+)ELi(\d+)ELb([01])E", n)
        if m:
            small.add(tuple(map(int, m.groups())))
        m = re.search(r"span_cta_kernelILb([01])ELi(\d+)ELi(\d+)ELi(\d+)E", n)
        if m:
            cta.add(tuple(map(int, m.groups())))
    assert small == set(SMALL_VARIANTS), (sorted(small - set(SMALL_VARIANTS)), sorted(set(SMALL_VARIANTS) - small))
    assert cta == set(CTA_VARIANTS), (sorted(cta - set(CTA_VARIANTS)), sorted(set(CTA_VARIANTS) - cta))
    assert len(small) + len(cta) == 40


# ---------------------------------------------------------------- the lab: stores, candidates, oracle
NX, NY, D = 256, 107, 2.0       # 107 rows: a prime, so every forced band height leaves a partial last band
WNX, WNY, WD = 1500, 23, 1.0    # chords of up to 47 words on a few rows
SEP = 15.0
POOL = 400_000                  # the batch-size ladder runs up to here
LADDER = sorted({int(round(128 * 1.04 ** k)) for k in range(400) if 128 * 1.04 ** k <= POOL})


def _candidates(rng, B, N, nx, ny, d):
    ex, ey = nx * d, ny * d
    X = np.concatenate([rng.random((B, N)) * (ex + 40) - 20, rng.random((B, N)) * (ey + 40) - 20,
                        (2 + rng.random((B, N)) * 28) * T], axis=1)
    k = rng.random(B)
    m = k < 0.15
    X[m] = np.rint(X[m])                                           # integer mesh: exact ties
    m = (k >= 0.15) & (k < 0.3)
    X[m, :2 * N] = np.rint(X[m, :2 * N] / (d / 2)) * (d / 2)      # centres on lattice lines and cell centres
    X[m, 2 * N:] = np.rint(X[m, 2 * N:] / d) * d                  # radii that are multiples of the pitch
    m = (k >= 0.3) & (k < 0.4)
    X[m, 2 * N:] *= 4                                              # tall discs
    X[:, N:2 * N][rng.random((B, N)) < 0.03] = -1e3                # discs off the grid
    X[:, 2 * N:][rng.random((B, N)) < 0.03] = 0.0                  # zero radius
    return X


def _near_boundary_discs(rng, n, nx, ny, d):
    """Centres placed so that the radicand of some cell is within a few ulps of T(R) (as in the parity suite)."""
    out = []
    for _ in range(n):
        i, j = int(rng.integers(1, nx + 1)), int(rng.integers(1, ny + 1))
        px, py = i * d - d / 2, j * d - d / 2
        R = float((2 + rng.random() * 28) * T) if rng.random() < 0.7 else float(rng.integers(1, 40)) * d
        th = rng.random() * 2 * math.pi if rng.random() < 0.6 else rng.choice([0, math.pi / 2, math.pi])
        cx, cy = px - R * math.cos(th), py - R * math.sin(th)
        for _ in range(int(rng.integers(0, 4))):
            cx = math.nextafter(cx, cx + rng.choice([-1.0, 1.0]))
        out.append((cx, cy, R))
    return out


def _band_candidates(rng, N=5):
    """Discs whose first or last covered row is a band's first or last row for every band height the tests force,
    discs taller than several bands, discs covering every row, discs off the grid, zero radii, near-boundary
    radicands; shuffled into candidates of N discs, plus a block of overlapping pairs."""
    discs = []
    edges = set()
    for h in (1, 4, 5, 16, 17, 32, 33):
        for jb0 in range(1, NY + 1, h):
            edges.add(jb0)
            edges.add(min(NY, jb0 + h - 1))
    for r in sorted(edges):
        for side in (-1, 1):  # -1: r is the disc's last covered row, +1: its first
            m = int(rng.integers(1, 25))
            cy = (r + side * m) * D - D / 2
            cx = int(rng.integers(1, NX + 1)) * D - D / 2
            for R in (m * D, math.nextafter(m * D, 0.0), math.nextafter(m * D, math.inf)):
                discs.append((cx, cy, R))
    for _ in range(300):  # taller than several bands
        discs.append((rng.random() * NX * D, rng.random() * NY * D, 30 + rng.random() * 120))
    for _ in range(40):   # every row (and every cell)
        discs.append((NX * D / 2 + rng.random() * 4, NY * D / 2 + rng.random() * 4, 300.0))
    for _ in range(150):  # off the grid, just beyond each edge
        R = 5 + rng.random() * 30
        discs.append(rng.choice([(-R - 1.0, rng.random() * NY * D, R), (NX * D + R + 1.0, rng.random() * NY * D, R),
                                 (rng.random() * NX * D, -R - 1.0, R), (rng.random() * NX * D, NY * D + R + 1.0, R)]))
    for _ in range(150):
        discs.append((rng.random() * NX * D, rng.random() * NY * D, 0.0))
    discs += _near_boundary_discs(rng, 1500, NX, NY, D)
    discs = np.array(discs)
    discs = discs[rng.permutation(len(discs))]
    discs = discs[:len(discs) // N * N].reshape(-1, N, 3)
    X = np.concatenate([discs[:, :, 0], discs[:, :, 1], discs[:, :, 2]], axis=1)
    pair = X[:150].copy()  # disc 1 = disc 0 one ulp smaller: the union, not the sum
    pair[:, 1], pair[:, N + 1] = pair[:, 0], pair[:, N]
    pair[:, 2 * N + 1] = np.nextafter(pair[:, 2 * N], 0.0)
    return np.concatenate([X, pair, _candidates(rng, 1000, N, NX, NY, D)])


class Lab:
    def __init__(self, cov, orc):
        self.cov, self.orc = cov, orc
        self.eng = cov.CoverageEngine(0)
        rng = np.random.default_rng(20261020)
        fire = rng.random((NX, NY)) < 0.1
        self.bits = cov.synth.pack_bits(fire)
        single = cov.synth.points_from_bits(self.bits, NX, D, D)
        # the multi-plane store: the same cells, 1-3 list entries each, two dyadic weight classes, list order shuffled
        mult = rng.integers(1, 4, len(single))
        w = np.where(rng.random(len(single)) < 0.5, 25.0, 100.0)
        multi = np.repeat(single, mult, axis=0)
        multi[:, 2] = multi[:, 3] = np.repeat(w, mult)
        multi = multi[rng.permutation(len(multi))]
        wfire = rng.random((WNX, WNY)) < 0.3
        self.wbits = cov.synth.pack_bits(wfire)
        self.pts = {"single": single, "multi": multi, "wide": cov.synth.points_from_bits(self.wbits, WNX, WD, WD)}
        self.store = None
        self.pools, self.want_cache, self.batches = {}, {}, {}

    def set_store(self, store):
        if store == self.store:
            return
        e = self.eng
        if store == "single":
            e.set_grid_bits(self.bits, NX, NY, D, D)
        elif store == "multi":
            e.set_points(self.pts["multi"], NX, NY, D, D)
        else:
            e.set_grid_bits(self.wbits, WNX, WNY, WD, WD)
        info = e.grid_info()
        assert info["area_exact"] == 1  # else every launch would go to the ordered kernel
        assert info["n_entries"] == len(self.pts[store])
        if store == "multi":
            assert info["n_classes"] == 2 and info["n_planes"] > 1
            self.class_w = e.class_weights()
        self.store = store

    def setup(self, store, N, kernel, fe=0, warps=0, ctas=0, band=0, mode=-1):
        self.set_store(store)
        self.eng.set_params(N, np.full(N, 30 * T), sep_min=SEP)
        c = self.cov
        for opt, v in ((c.OPT_KERNEL, kernel), (c.OPT_FORCE_EXACT, fe), (c.OPT_WARPS_PER_CTA, warps),
                       (c.OPT_CTAS_PER_SM, ctas), (c.OPT_BAND_ROWS, band), (c.OPT_PLANE_MODE, mode)):
            self.eng.set_option(opt, v)

    def pool(self, name, N):
        if (name, N) not in self.pools:
            rng = np.random.default_rng(1000 + N)
            if name == "random":
                X = _candidates(rng, POOL if N <= 8 else 400, N, NX, NY, D)
            elif name == "band":
                X = _band_candidates(rng, N)
            else:  # wide: chords of 19 to 47 words beside narrow discs
                B = 1200
                X = np.concatenate([rng.random((B, N)) * WNX * WD, rng.random((B, N)) * (WNY + 10) - 5,
                                    np.where(rng.random((B, N)) < 0.6, 300 + rng.random((B, N)) * 600,
                                             rng.random((B, N)) * 50)], axis=1)
                X[:100, :N] = WNX * WD / 2 + rng.random((100, N)) * 10  # centred: chords across the whole grid
                X[:100, 2 * N:] = 700 + rng.random((100, N)) * 100
            self.pools[name, N] = X
        return self.pools[name, N]

    def want(self, store, name, N, B):
        """Oracle results for the first B candidates of a pool (extended on demand: rows are independent)."""
        key = (store, name, N)
        self.set_store(store)  # (the class numbering of the multi-plane store)
        X = self.pool(name, N)
        have = self.want_cache.get(key)
        n0 = 0 if have is None else len(have["obj"])
        if B > n0:
            pts = self.pts[store]
            part = self.orc.eval_batch(X[n0:B], N, np.full(N, 30 * T), pts, want_prog=True, sep_min=SEP)
            if store == "multi":  # class 0 from its own entries, class 1 the rest
                c0 = self.orc.eval_batch(X[n0:B], N, np.full(N, 30 * T), pts[pts[:, 3] == self.class_w[0]])["count"]
                part["class_count"] = np.stack([c0, part["count"] - c0], axis=1)
            have = part if have is None else {k: np.concatenate([have[k], part[k]]) for k in part}
            self.want_cache[key] = have
        return {k: v[:B] for k, v in have.items()}

    def small_batches(self, store, N, cap):
        """{(chunk, max_warps): B} for the small-swarm kernel on this store: a geometric ladder of batch sizes is
        probed on the device (the choice depends on the SM count and the warps that fit), then each found B is moved
        to a ragged one (B = 1 or CHUNK - 1 mod CHUNK) that still selects the same instantiation."""
        key = (store, N, cap)
        if key in self.batches:
            return self.batches[key]
        e, K = self.eng, self.cov.KERNEL_SPAN
        self.setup(store, N, kernel=K, warps=cap)
        X = self.pool("random", N)
        dX, d_obj = e.device_alloc(X.nbytes), e.device_alloc(len(X) * 8)
        try:
            e.memcpy_h2d(dX, X)

            def probe(B):
                e.eval_batch_device(dX, B, d_obj)
                li = e.last_launch()
                return (li["chunk"], li["max_warps"]) if li["kernel"] == K else None

            seen = {}
            for B in LADDER:
                seen.setdefault(probe(B), []).append(B)
            found = {}
            for sel, Bs in seen.items():
                if sel is None:
                    continue
                # (batches up to one host-path slice of ~16 MiB: the real run must be a single launch)
                Bs = [b for b in Bs if b * 24 * N <= (16 << 20)] or Bs[:1]
                c, mid = sel[0], Bs[len(Bs) // 2]
                base = mid // c * c
                for B in (base + 1, base + c - 1, base - c + 1, base - 1, base + c + 1, base - 2 * c + 1):
                    if 128 <= B <= len(X) and probe(B) == sel:
                        found[sel] = B
                        break
            e.sync()
        finally:
            e.device_free(dX)
            e.device_free(d_obj)
        self.batches[key] = found
        return found

    def check(self, got, want, rows="all"):
        for k in ("count", "feasible"):
            bad = np.flatnonzero(got[k] != want[k])
            assert bad.size == 0, (rows, k, bad[:10], got[k][bad[:5]], want[k][bad[:5]])
        for k in ("obj", "progressive"):
            bad = np.flatnonzero(got[k].view(np.uint64) != want[k].view(np.uint64))
            assert bad.size == 0, (rows, k, bad[:10], got[k][bad[:5]], want[k][bad[:5]])
        if "class_count" in want:
            bad = np.flatnonzero((got["class_count"] != want["class_count"]).any(axis=1))
            assert bad.size == 0, (rows, "class_count", bad[:10])

    def run(self, store, name, N, B):
        X = self.pool(name, N)[:B]
        got = self.eng.eval_batch(X, want_progressive=True, want_class_count=store == "multi")
        return got, self.eng.last_launch()

    def close(self):
        self.eng.close()


@pytest.fixture(scope="module")
def lab(cov, orc):
    lb = Lab(cov, orc)
    yield lb
    lb.close()


# ---------------------------------------------------------------- GPU: every instantiation against the oracle
def _small_id(v):
    return "multi%d-chunk%d-maxw%d-few%d" % v


@pytest.mark.gpu
@pytest.mark.parametrize("variant", SMALL_VARIANTS, ids=_small_id)
def test_small_kernel_instantiation_vs_oracle(cov, lab, variant):
    multi, chunk, maxw, few = variant
    N = 5 if few else (7 if maxw == 24 else 6)   # FEW is N <= 5; N = 6 and 7 take the general disc lookup
    cap = 20 if maxw == 20 else 0                # COV_OPT_WARPS_PER_CTA: at most 20 warps
    store = "multi" if multi else "single"
    found = lab.small_batches(store, N, cap)
    assert (chunk, maxw) in found, f"no batch size selects chunk {chunk} / {maxw} warps; reachable: {sorted(found)}"
    B = found[chunk, maxw]
    assert B % chunk in (1, chunk - 1)           # the last unit is ragged
    want = lab.want(store, "random", N, B)
    for fe in (0, 1):
        lab.setup(store, N, kernel=cov.KERNEL_SPAN, fe=fe, warps=cap)
        got, li = lab.run(store, "random", N, B)
        assert (li["kernel"], li["multi"], li["chunk"], li["max_warps"]) == (cov.KERNEL_SPAN, multi, chunk, maxw), li
        assert (20 if maxw == 24 else 0) * 32 < li["block"] <= maxw * 32, li
        lab.check(got, want, (variant, B, fe))


def _cta_id(v):
    return "multi%d-mode%d-threads%d-ctas%d" % v


@pytest.mark.gpu
@pytest.mark.parametrize("variant", CTA_VARIANTS, ids=_cta_id)
def test_cta_kernel_instantiation_vs_oracle(cov, lab, variant):
    multi, mode, threads, ctas = variant
    r = CTA_REACH[variant]
    N = r["N"]
    B = 2501 if N <= 8 else 301
    store = "multi" if multi else "single"
    want = lab.want(store, "random", N, B)
    for fe in (0, 1):
        lab.setup(store, N, kernel=cov.KERNEL_SPAN_GENERAL, fe=fe, ctas=r.get("ctas", 0), mode=r["mode"])
        got, li = lab.run(store, "random", N, B)
        assert (li["kernel"], li["multi"], li["plane_mode"], li["block"], li["chunk"]) == \
            (cov.KERNEL_SPAN_GENERAL, multi, mode, threads, ctas), li
        assert li["planes_in_smem"] == (mode in (2, 3))
        lab.check(got, want, (variant, fe))


# ---------------------------------------------------------------- GPU: band and unit edges of the CTA kernel
BAND_MODES = {"mode0": ("single", 0), "mode1": ("single", 1), "mode2": ("single", 2), "mode3": ("single", 3),
              "mode4": ("single", 4), "multi": ("multi", -1)}


@pytest.mark.gpu
@pytest.mark.parametrize("which", list(BAND_MODES))
def test_cta_kernel_band_edges_vs_oracle(cov, lab, which):
    store, mode = BAND_MODES[which]
    aligned = mode in (2, 3, 4)                  # TMA / sweep bands start on 16-byte boundaries of the plane
    N = 5
    B = len(lab.pool("band", N))
    want = lab.want(store, "band", N, B)
    for v in (0, 4 if aligned else 1, 5, 17, 33):
        for fe in (0, 1):
            lab.setup(store, N, kernel=cov.KERNEL_SPAN_GENERAL, fe=fe, band=v, mode=mode)
            got, li = lab.run(store, "band", N, B)
            assert li["kernel"] == cov.KERNEL_SPAN_GENERAL and li["plane_mode"] == max(mode, 0), li
            rows = NY if v == 0 else (max(4, v & ~3) if aligned else v)
            assert li["band_rows"] == rows, (v, li)
            lab.check(got, want, (which, v, fe))


@pytest.mark.gpu
def test_wide_chords_vs_oracle(cov, lab):
    """nx = 1500: chords of up to 47 words run the whole-word loops of paint_only (sweep modes) and paint_span
    (the small-swarm kernel and the early mode) past their unrolled part."""
    N = 5
    B = len(lab.pool("wide", N))
    want = lab.want("wide", "wide", N, B)
    runs = [(cov.KERNEL_SPAN, -1, 0, cov.KERNEL_SPAN)] + \
        [(cov.KERNEL_SPAN_GENERAL, m, band, cov.KERNEL_SPAN_GENERAL) for m in (1, 3, 4) for band in (0, 5)]
    for kernel, mode, band, ran in runs:
        for fe in (0, 1):
            lab.setup("wide", N, kernel=kernel, fe=fe, band=band, mode=mode)
            got, li = lab.run("wide", "wide", N, B)
            assert li["kernel"] == ran and (mode < 0 or li["plane_mode"] == mode), li
            lab.check(got, want, (kernel, mode, band, fe))
    assert want["count"].max() > 0.9 * len(lab.pts["wide"])
