"""hnanosolver_b200: B200-native (sm_100a) implementation of HNanoSolver's per-frame sparse fluid step.

The package holds only what the hot path needs: the CUDA kernels + C ABI (csrc/, built into libhns_b200.so) and the
host-side mirror of the reference's launcher interface (launchers.py, grid_data.py). There is no CPU fallback.
"""
from .grid_data import FLOAT, VEC3F, AllocationType, GridIndexedData  # noqa: F401
from ._lib import CombustionParams, HnsError, HnsInvalidArgument  # noqa: F401
from .launchers import (AdvectIndexGrid, AdvectIndexGridVelocity, CombustionKernel, Compute_Sim, CreateIndexGrid,  # noqa: F401
                        Divergence, IndexGridHandle, Multigrid, ProjectNonDivergent, Simulation, Source, ValueGrid, build_domain,
                        create_index_grid_from_origins)
