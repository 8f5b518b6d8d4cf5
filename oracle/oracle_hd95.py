"""CPU restatement of the HD95 surface distance.  TEST INFRASTRUCTURE ONLY (oracle).

``surface_distances`` / ``hd95`` restate medpy's ``__surface_distances`` and ``hd95`` (connectivity 1), the reference's
medpy-based metric module, with scipy.ndimage and numpy.percentile.  medpy raises on an empty mask; these give an empty
array / NaN.  The Dice oracle is oracle_metric.py.
PARITY PIN: tests/test_oracle_hd95.py checks it against known answers and a brute-force restatement.
"""
from __future__ import annotations

import numpy as np
from scipy.ndimage import binary_erosion, distance_transform_edt, generate_binary_structure


def border(mask: np.ndarray) -> np.ndarray:
    """mask ^ binary_erosion(mask, 6-connected), the outside of the volume counted as background."""
    return mask ^ binary_erosion(mask, structure=generate_binary_structure(mask.ndim, 1), iterations=1)


def surface_distances(result, reference, spacing=None) -> np.ndarray:
    """medpy ``__surface_distances(result, reference, voxelspacing, connectivity=1)``: for every border voxel of
    ``result`` the distance to the nearest border voxel of ``reference``.  Empty float64 array when either mask is
    empty."""
    result = np.atleast_1d(np.asarray(result).astype(bool))
    reference = np.atleast_1d(np.asarray(reference).astype(bool))
    if not result.any() or not reference.any():
        return np.zeros(0, dtype=np.float64)
    if spacing is not None:
        spacing = np.asarray(spacing, dtype=np.float64)
    dt = distance_transform_edt(~border(reference), sampling=spacing)
    return dt[border(result)]


def hd95(result, reference, spacing=None) -> float:
    """medpy ``hd95(result, reference, voxelspacing, connectivity=1)``; NaN when either mask is empty."""
    d_ab = surface_distances(result, reference, spacing)
    d_ba = surface_distances(reference, result, spacing)
    if d_ab.size == 0 or d_ba.size == 0:
        return float("nan")
    return float(np.percentile(np.hstack((d_ab, d_ba)), 95))
