"""Pins the HD95 oracle (oracle/oracle_hd95.py: surface_distances, hd95) against known answers and against an
independent brute-force restatement: explicit 6-neighbour borders, the minimum over all border-voxel pairs, and the
percentile's linear interpolation written out."""
import math

import numpy as np
import pytest

from oracle import oracle_hd95


def _border_brute(m):
    p = np.pad(m, 1, constant_values=False)
    inner = np.ones_like(m)
    D, H, W = m.shape
    for dz, dy, dx in ((1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)):
        inner &= p[1 + dz:1 + dz + D, 1 + dy:1 + dy + H, 1 + dx:1 + dx + W]
    return m & ~inner


def _dist_brute(a, b, s):
    pa, pb = np.argwhere(_border_brute(a)), np.argwhere(_border_brute(b))
    t = (pb[None, :, :] - pa[:, None, :]).astype(np.float64) * np.asarray(s, dtype=np.float64)
    t = t * t
    return np.sqrt((t[..., 0] + t[..., 1]) + t[..., 2]).min(axis=1)


def _hd95_brute(a, b, s=(1.0, 1.0, 1.0)):
    if not a.any() or not b.any():
        return float("nan")
    x = np.sort(np.concatenate([_dist_brute(a, b, s), _dist_brute(b, a, s)]))
    n = len(x)
    h = (n - 1) * 0.95
    lo = math.floor(h)
    hi = min(lo + 1, n - 1)
    g = h - lo
    d = x[hi] - x[lo]
    return float(x[hi] - d * (1 - g)) if g >= 0.5 else float(x[lo] + d * g)


def _cube(shape, lo, hi):
    m = np.zeros(shape, dtype=bool)
    m[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] = True
    return m


def test_identical_masks_give_zero():
    m = _cube((9, 10, 11), (2, 3, 1), (7, 8, 6))
    assert oracle_hd95.hd95(m, m) == 0.0
    assert oracle_hd95.hd95(m, m, (2.0, 1.5, 1.5)) == 0.0


def test_single_voxels_at_a_known_offset():
    a, b = np.zeros((8, 8, 8), dtype=bool), np.zeros((8, 8, 8), dtype=bool)
    a[1, 1, 2] = True
    b[4, 5, 2] = True  # offset (3, 4, 0)
    assert oracle_hd95.hd95(a, b) == 5.0
    assert oracle_hd95.hd95(a, b, (2.0, 1.0, 1.0)) == math.sqrt(52.0)
    assert oracle_hd95.surface_distances(a, b, (2.0, 1.0, 1.0)).tolist() == [math.sqrt(52.0)]


def test_full_volume_mask_has_only_its_outer_shell_as_border():
    full = np.ones((5, 6, 7), dtype=bool)
    shell = np.ones_like(full)
    shell[1:-1, 1:-1, 1:-1] = False
    assert np.array_equal(oracle_hd95.border(full), shell)
    assert np.array_equal(_border_brute(full), shell)
    assert oracle_hd95.surface_distances(full, full).shape == (int(shell.sum()),)


def test_one_voxel_thick_sheet_is_all_border():
    sheet = _cube((6, 9, 9), (3, 1, 1), (4, 8, 8))
    assert np.array_equal(oracle_hd95.border(sheet), sheet)
    assert np.array_equal(_border_brute(sheet), sheet)


@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("spacing", [(1.0, 1.0, 1.0), (2.0, 1.5, 1.5), (0.5, 1.25, 3.0)])
def test_shifted_cubes_match_the_brute_force(axis, spacing):
    lo, hi = [2, 3, 1], [6, 8, 5]
    a = _cube((10, 12, 11), lo, hi)
    lo[axis] += 2
    hi[axis] += 3
    b = _cube((10, 12, 11), lo, hi)
    b[lo[0] + 1, lo[1] + 1, lo[2] + 1] = False  # a cavity: an inner border
    exp = _hd95_brute(a, b, spacing)
    assert exp > 0
    assert oracle_hd95.hd95(a, b, spacing) == exp  # squared terms exact in fp64: same bits
    assert oracle_hd95.hd95(b, a, spacing) == exp


def test_random_blobs_match_the_brute_force():
    rng = np.random.default_rng(3)
    a = rng.random((7, 9, 8)) > 0.6
    b = rng.random((7, 9, 8)) > 0.7
    for s in ((1.0, 1.0, 1.0), (2.0, 1.5, 1.5)):
        assert oracle_hd95.hd95(a, b, s) == _hd95_brute(a, b, s)
    assert oracle_hd95.hd95(a, b, (0.7, 0.8, 2.5)) == pytest.approx(_hd95_brute(a, b, (0.7, 0.8, 2.5)), rel=1e-12)


def test_empty_masks_give_nan():
    m = _cube((6, 6, 6), (1, 1, 1), (4, 4, 4))
    z = np.zeros_like(m)
    assert math.isnan(oracle_hd95.hd95(z, m))
    assert math.isnan(oracle_hd95.hd95(m, z))
    assert math.isnan(oracle_hd95.hd95(z, z))
    assert oracle_hd95.surface_distances(z, m).size == 0
