"""libcoverage_cuda -- B200-native (sm_100a) batched coverage objective for UAV-swarm MADS
optimisation, with a host-side mirror of the reference's interface for that path.

The directory name contains a dot, so import it through the alias module at the repo root:

    import coverage_b200 as cov
    cells = cov.CellFunctions.initialise_POI(cov.CellFunctions.Cells(), "static")
    obj = cov.TDM_STATIC_opt.createObjective(cells, 5, r_max)
    obj(x); obj.batch(X)

Importing this package loads libcoverage_cuda.so and raises if it is missing (no CPU fallback).
"""
from . import _lib  # noqa: F401  (loads the shared library; raises ImportError when absent)
from ._lib import CoverageError, KERNEL_AUTO, KERNEL_SPAN, KERNEL_BRUTE, KERNEL_EXACT, KERNEL_SPAN_GENERAL, KERNEL_ORDERED  # noqa: F401
from ._lib import OPT_KERNEL, OPT_WARPS_PER_CTA, OPT_CTAS_PER_SM, OPT_BAND_ROWS, OPT_FORCE_EXACT, OPT_CHUNK, OPT_TRACE, OPT_ZEROCOPY_OUT, OPT_PLANE_MODE, OPT_PROGRESSIVE_INDEX, OPT_LIST_ORDER_HORIZON  # noqa: F401
from ._lib import PACK_F32, PACK_I32, PACK_I16  # noqa: F401
from .engine import CoverageEngine, TAN_HALF_FOV_DEFAULT, threshold, limits, device_count, pack_candidates  # noqa: F401
from . import AreaCoverageCalculation, CellFunctions, TDM_Constraints, TDM_STATIC_opt, Base_Functions  # noqa: F401
from . import fire_io, synth, mads, FullSimulation, DynamicArea  # noqa: F401

__all__ = ["CoverageEngine", "CoverageError", "AreaCoverageCalculation", "CellFunctions", "TDM_Constraints",
           "TDM_STATIC_opt", "Base_Functions", "FullSimulation", "DynamicArea", "mads", "fire_io", "synth", "threshold", "limits", "device_count"]
