"""The SDF query restatement for either ScalarType (TEST INFRASTRUCTURE ONLY).

``sdf_queries_oracle.SdfOracle`` restates the reference's SignedDistanceField<float> queries and
stores the field as float32. ``SdfOracle`` here is the same restatement, every method inherited,
with the field stored as ``dtype``: float32 by default (then it is the float oracle), float64 for
SignedDistanceField<double>. The restatement computes on numpy scalars of the stored type, so
the statements where the reference computes in ScalarType become double arithmetic by
themselves for float64:

    include/voxelized_geometry_tools/signed_distance_field.hpp
      :932-943   the interior coarse gradient's difference of two neighbours (a double
                 subtraction, then times the double 1 / (2 * resolution))
      :494-534   GetNextFromGradient's sign test of the cell (< 0.0 on the double value)

Everything else already reads a cell as a double and stays in double. A double cell is never
rounded through float: -1e-300 stays negative, 1.0 - 1e-9 stays below 1.0.

PARITY STATUS. The float statements are pinned against the reference's own members
(tests/test_sdf_queries_vs_reference.py, where oracle/_ref is built); the double instantiation
is restated from them and is not pinned against the reference's own SignedDistanceField<double>.
"""
from __future__ import annotations

import numpy as np

from .sdf_queries_oracle import NO_VALUE, THROWS, VALUE  # noqa: F401  (re-exported)
from . import sdf_queries_oracle

SCALAR_TYPES = (np.dtype(np.float32), np.dtype(np.float64))


class SdfOracle(sdf_queries_oracle.SdfOracle):
    def __init__(self, sdf: np.ndarray, resolution: float, origin_transform=None,
                 dtype=np.float32):
        dtype = np.dtype(dtype)
        if dtype not in SCALAR_TYPES:
            raise ValueError(f"the SDF's scalar type is float32 or float64, not {dtype}")
        # the base sets the frames and the dimensions; the field it stores is then replaced
        super().__init__(np.zeros(np.shape(sdf), dtype=np.float32), resolution, origin_transform)
        self.sdf = np.ascontiguousarray(sdf, dtype=dtype)
