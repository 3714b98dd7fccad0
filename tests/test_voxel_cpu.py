"""The voxeliser's CPU restatement (oracle/voxel_oracle.c) against analytic shapes and its tie rules."""
import sys
from pathlib import Path

import numpy as np
import pytest

import helpers as H

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import oracle as O  # noqa: E402


def centres(n, o, h):
    return o + (np.arange(n) + 0.5) * h


def test_box_with_rays_through_shared_edges():
    """every face of the box is split along a diagonal and the rays of the rows with j == k run
    exactly through those diagonals (and through the box's corners' projections): each crossing must
    count once"""
    tri = H.mesh_box((1.0, 1.0, 1.0), (5.0, 5.0, 5.0))
    m = O.voxelize(tri, (0.0, 0.0, 0.0), 0.5, (12, 12, 12))
    c = centres(12, 0.0, 0.5)
    inside = (c > 1.0) & (c < 5.0)
    expect = inside[:, None, None] & inside[None, :, None] & inside[None, None, :]
    assert np.array_equal(m.astype(bool), expect)
    # centres exactly ON the faces y = 1 / z = 5 (grid shifted by a quarter voxel): still a clean box
    m2 = O.voxelize(tri, (0.25, 0.25, 0.25), 0.5, (12, 12, 12))
    c2 = centres(12, 0.25, 0.5)
    assert set(np.unique(m2.sum(axis=2))) <= {0, int(((c2 > 1.0) & (c2 < 5.0)).sum()), int(((c2 >= 1.0) & (c2 < 5.0)).sum())}
    assert m2.sum() > 0 and m2[:, :, 0].sum() == 0 and m2[:, :, -1].sum() == 0


@pytest.mark.parametrize("h", [0.5, 0.31])
def test_sphere_matches_the_analytic_inside_test_up_to_the_surface(h):
    ctr, r = np.array([8.1, 7.9, 8.3]), 6.0
    tri = H.mesh_sphere(ctr, r, nu=96, nv=48)
    n = int(16.5 / h)
    m = O.voxelize(tri, (0.0, 0.0, 0.0), h, (n, n, n)).astype(bool)
    c = centres(n, 0.0, h)
    d = np.sqrt((c[None, None, :] - ctr[0]) ** 2 + (c[None, :, None] - ctr[1]) ** 2 + (c[:, None, None] - ctr[2]) ** 2)
    # the faceted sphere lies within r*(1-cos(pi/48)) of the true one: no disagreement outside that shell
    tol = r * (1 - np.cos(np.pi / 48)) + 1e-6
    assert not (m & (d > r + 1e-6)).any()
    assert not (~m & (d < r - tol)).any()
    assert abs(m.sum() * h ** 3 / (4 / 3 * np.pi * r ** 3) - 1) < 0.02


def test_open_tube_slabs_and_triangle_order():
    tri = H.mesh_tube(20.0, 3.0, bend=1.5, x0=6.0, z0=5.0)
    grid = ((0.0, 0.0, 0.0), 0.25, (48, 80, 40))
    m = O.voxelize(tri, *grid)
    assert m[:, 0, :].sum() > 0 and m[:, -1, :].sum() > 0  # open ends along y are filled too
    # z-slabs tile the full result
    parts = [O.voxelize(tri, *grid, z_range=r) for r in ((0, 13), (13, 14), (14, 40))]
    assert np.array_equal(np.concatenate(parts), m)
    # order-independent
    rng = np.random.default_rng(0)
    assert np.array_equal(O.voxelize(tri[rng.permutation(len(tri))], *grid), m)
    # cross-section area of plane y ~ pi r^2
    area = m[:, 40, :].sum() * 0.25 ** 2
    assert abs(area / (np.pi * 9.0) - 1) < 0.03


def test_rows_through_a_ragged_rim_are_cleared():
    """triangles missing at an open end: rays that meet only one wall there have no inside/outside
    answer; such rows come out empty instead of painted to the edge of the box"""
    tri = H.mesh_tube(20.0, 3.0, x0=6.0, z0=5.0)
    ragged = np.delete(tri, np.arange(len(tri) - 40, len(tri) - 10), axis=0)  # a hole in the last ring, one side only
    grid = ((0.0, 0.0, 0.0), 0.25, (48, 80, 40))
    full, m = O.voxelize(tri, *grid), O.voxelize(ragged, *grid)
    assert m[:, :, -1].sum() == 0 and m[:, :, 0].sum() == 0   # nothing leaks to the box edge
    assert np.array_equal(m[:, :78], full[:, :78])             # rows away from the hole are untouched
    assert 0 < m[:, 78:].sum() < full[:, 78:].sum()            # rows through the hole are cleared

