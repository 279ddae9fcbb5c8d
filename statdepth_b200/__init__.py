"""statdepth_b200 -- B200-native drop-in for statdepth's depth hot path.

    from statdepth_b200 import FunctionalDepth, PointcloudDepth      # == from statdepth import ...
    from statdepth_b200 import FunctionalDepthOf, PointcloudDepthOf  # depth of new data against a reference sample
    from statdepth_b200 import FunctionalBoxplot, Outliergram        # functional outlier detection
    from statdepth_b200 import ExtremalDepth                         # extremal depth (Narisetty & Nair 2016)
    from statdepth_b200 import HalfspaceDepth, FunctionalHalfspaceDepth  # halfspace (Tukey) depth, d = 1 or 2
    from statdepth_b200 import ProjectionDepth, FunctionalProjectionDepth  # random projection depths, any d
    from statdepth_b200 import FunctionalReference, DepthClassifier  # a reference fitted once; max-depth classes
    from statdepth_b200 import FunctionalProjectionDepthOf, ProjectionDepthOf  # projection depths of new data
    from statdepth_b200 import FunctionalSpatialDepth, FunctionalSpatialDepthOf  # L2 spatial depth of curves
    from statdepth_b200 import FunctionalModalDepth, FunctionalModalDepthOf  # h-modal (kernel) depth of curves
    from statdepth_b200 import FunctionalKernelSpatialDepth, FunctionalKernelSpatialDepthOf  # KFSD of curves
    from statdepth_b200.homogeneity import FunctionalHomogeneity     # == statdepth.homogeneity
    from statdepth_b200.testing import generate_noisy_univariate     # == statdepth.testing

All depth arithmetic runs in hand-written sm_100a CUDA kernels behind the C ABI declared in
include/statdepth_b200.h (libsdepth.so, loaded with ctypes).  There is no CPU fallback: without the
library or without a B200 every depth call raises `EngineUnavailable`.  Multi-GPU sharding of a call (one process
per GPU, torch.distributed) is opt-in: `enable_distributed()`, see _dist.py.
"""
from ._dist import enable_distributed
from ._engine import Engine, EngineError, EngineUnavailable, get_engine
from ._helper import DepthDegeneracy
from .depth import (DepthClassifier, ExtremalDepth, FunctionalBoxplot, FunctionalDepth, FunctionalDepthOf,
                    FunctionalHalfspaceDepth, FunctionalKernelSpatialDepth, FunctionalKernelSpatialDepthOf,
                    FunctionalProjectionDepth, FunctionalProjectionDepthOf,
                    FunctionalModalDepth, FunctionalModalDepthOf, FunctionalReference, FunctionalSpatialDepth,
                    FunctionalSpatialDepthOf, HalfspaceDepth, Outliergram, PointcloudDepth, PointcloudDepthOf,
                    ProjectionDepth, ProjectionDepthOf)
from .settings import get_simplex_tolerance, set_simplex_tolerance

__version__ = "0.1.0"
__all__ = ["FunctionalDepth", "PointcloudDepth", "FunctionalDepthOf", "PointcloudDepthOf", "FunctionalBoxplot",
           "Outliergram", "ExtremalDepth", "HalfspaceDepth", "FunctionalHalfspaceDepth", "ProjectionDepth", "FunctionalProjectionDepth", "FunctionalReference", "DepthClassifier", "FunctionalProjectionDepthOf", "ProjectionDepthOf", "FunctionalSpatialDepth", "FunctionalSpatialDepthOf", "FunctionalModalDepth", "FunctionalModalDepthOf", "FunctionalKernelSpatialDepth", "FunctionalKernelSpatialDepthOf", "DepthDegeneracy", "Engine", "EngineError", "EngineUnavailable",
           "get_engine", "get_simplex_tolerance", "set_simplex_tolerance", "enable_distributed"]
