"""CPU-only: what nvcc built.  The library must carry sm_100a code only, its objective kernels must fit the occupancy
their launchers plan for (registers per thread, no local-memory arrays), and the fire-plane staging must really be
TMA bulk copies completing on mbarriers (UBLKCP / SYNCS in the SASS) -- read with cuobjdump, no GPU needed."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "maximumareacoverageoptimization.jl_b200", "libcoverage_cuda.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"

pytestmark = pytest.mark.skipif(not (os.path.exists(CUOBJDUMP) and os.path.exists(LIB)),
                                reason="needs cuobjdump and the built library")


def _run(*args):
    return subprocess.run([CUOBJDUMP, *args, LIB], capture_output=True, text=True, timeout=300).stdout


@pytest.fixture(scope="module")
def usage():
    """mangled kernel name -> dict(REG, STACK, SHARED, LOCAL)"""
    out = {}
    name = None
    for line in _run("-res-usage").splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            out[name] = {k: int(v) for k, v in re.findall(r"(REG|STACK|SHARED|LOCAL):(\d+)", line)}
            name = None
    return out


def test_only_sm100a_code():
    elfs = [l for l in _run("-lelf").splitlines() if "ELF file" in l]
    assert elfs and all(l.rstrip().endswith(".sm_100a.cubin") for l in elfs), elfs
    assert "PTX file" not in _run("-lptx")  # nothing for a JIT to retarget: sm_100a or nothing


def test_objective_kernels_fit_their_launch_plans(usage):
    small = {k: v for k, v in usage.items() if "span_small_kernel" in k}
    cta = {k: v for k, v in usage.items() if "span_cta_kernel" in k}
    assert len(small) == 30 and len(cta) >= 8  # 2 x 4 x 2 x 2, less <*, 32, 24, false> (tests/test_launch_matrix.py)
    for k, v in {**small, **cta, **{k: v for k, v in usage.items() if re.search(r"brute_kernel|exact_kernel|ordered_kernel", k)}}.items():
        assert v["LOCAL"] == 0, (k, v)          # no local-memory arrays (the stack frame is the FP64 slow path's call)
        assert v["STACK"] <= 128, (k, v)
    for k, v in small.items():                  # span_small_kernel<MULTI, CHUNK, MAXW, FEW>: one CTA of MAXW warps per SM
        maxw = int(re.search(r"ILb[01]ELi\d+ELi(\d+)ELb[01]E", k).group(1))
        assert v["REG"] * 32 * maxw <= 65536, (k, v)
    for k, v in cta.items():                    # span_cta_kernel<MULTI, PLANES, THREADS, CTAS>: CTAS co-resident CTAs per SM
        threads, ctas = map(int, re.search(r"ILb[01]ELi\d+ELi(\d+)ELi(\d+)E", k).groups())
        assert v["REG"] * threads * ctas <= 65536, (k, v)


def test_plane_staging_is_tma_bulk_copy_on_mbarriers():
    """cp.async.bulk (UBLKCP) + mbarrier (SYNCS) in the span kernels' SASS; no tensor-core instructions anywhere
    (a mask / count workload, north_star)."""
    sass = _run("-sass")
    per_fn = re.split(r"\n\s*Function : ", sass)
    span = [f for f in per_fn if f.startswith("_ZN3cov17span_small_kernel") or f.startswith("_ZN3cov15span_cta_kernel")]
    assert span
    assert all("UBLKCP" in f and "SYNCS" in f for f in span if f.startswith("_ZN3cov17span_small_kernel"))
    assert any("UBLKCP" in f for f in span if f.startswith("_ZN3cov15span_cta_kernel"))
    assert not re.search(r"\b(HMMA|IMMA|QMMA|UTCHMMA|UTCQMMA|UTCIMMA)\b", sass)
