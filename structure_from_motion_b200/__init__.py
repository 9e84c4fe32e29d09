"""structure_from_motion_b200 — B200-native two-view geometry hot path.

RANSAC essential-matrix estimation (eight-point fits scored by symmetric epipolar distance)
-> cheirality vote -> linear triangulation, as hand-written sm_100a CUDA kernels behind a
C ABI (include/sfm_b200.h), mirrored here under the reference's Python signatures.
The reference's import paths (``lib.ransac.ransac``, ``lib.epipolar.*`` ...) are provided by
the top-level ``lib`` package, which aliases the sub-modules of this package.
"""
from .errors import EightPointCalculationError  # noqa: F401
from .model_selection import (  # noqa: F401
    ModelScores, TwoViewSelection, batch_two_view_select_arrays, model_scores_arrays, two_view_select_arrays)
from .ransac.ransac import ErrorAggregationMethod  # noqa: F401

__version__ = "0.1.0"
