"""The connected-component oracle (oracle/oracle_components.py, scipy.ndimage.label) against an independent breadth-first
flood fill, and on hand cases whose answer is known (CPU only)."""
import numpy as np
import pytest

import oracle_components as OC
import oracle_hausdorff as OH

CONNECTIVITIES = [("2d", 1), ("2d", 2), ("3d", 1), ("3d", 2), ("3d", 3)]


def assert_same(a, b):
    for x, y, name in zip(a, b, ("labels", "stats", "largest")):
        assert x.dtype == y.dtype and x.shape == y.shape, name
        assert np.array_equal(x, y), name


@pytest.mark.parametrize("method,conn", CONNECTIVITIES)
@pytest.mark.parametrize("shape,C", [((3, 9, 11), 2), ((2, 12, 7), 3), ((4, 6, 6), 4), ((1, 1, 13), 2), ((7, 1, 1), 2)])
def test_oracle_matches_flood_fill(shape, C, method, conn):
    rng = np.random.default_rng(C * 100 + shape[1])
    for kind in range(3):
        if kind == 0:
            m = OH.salt_pepper(rng, shape, C)
        elif kind == 1 and min(shape[1:]) > 2:
            m = OH.blobs(rng, shape, C, smooth=1.0)
        else:
            m = rng.choice(np.array([0, 1, C - 1, C, -2]), size=shape, p=[0.4, 0.3, 0.2, 0.05, 0.05])
        assert_same(OC.components(m, C, method, conn), OC.components_bfs(m, C, method, conn))


def test_tie_goes_to_the_first_component():
    m = np.zeros((1, 5, 9), np.int64)
    m[0, 3, 0:3] = 1      # first pixel index 27, size 3
    m[0, 0, 6:9] = 1      # first pixel index 6, size 3: first in raster order
    m[0, 2, 5] = 2
    m[0, 4, 8] = 2        # two single pixels of class 2
    for method, conn in CONNECTIVITIES[:2]:
        labels, stats, largest = OC.components(m, 3, method, conn)
        assert stats[0, 1].tolist() == [2, 3] and stats[0, 2].tolist() == [2, 1]
        want = np.zeros_like(m)
        want[0, 0, 6:9] = 1
        want[0, 2, 5] = 2
        assert np.array_equal(largest, want)
        assert labels[0, 3, 1] == 27 and labels[0, 0, 7] == 6 and labels[0, 4, 8] == 44
        assert_same((labels, stats, largest), OC.components_bfs(m, 3, method, conn))


def test_out_of_range_values_belong_to_no_component():
    m = np.zeros((2, 4, 4), np.int64)
    m[0, 1, 1] = 5; m[1, 2, 2] = -1; m[1, 0, 0] = 1; m[1, 3, 3] = 1
    for method, conn in CONNECTIVITIES:
        labels, stats, largest = OC.components(m, 2, method, conn)
        assert labels[0, 1, 1] == -1 and labels[1, 2, 2] == -1
        assert largest[0, 1, 1] == 5 and largest[1, 2, 2] == -1
        assert stats[..., 1].sum() <= 32 - 2
        assert np.array_equal(largest[1, 0, 0], 1) and largest[1, 3, 3] == 0
        assert_same((labels, stats, largest), OC.components_bfs(m, 2, method, conn))
    _, stats, _ = OC.components(m, 2, "2d", 1)
    assert stats[0, 0].tolist() == [1, 15] and stats[1, 0].tolist() == [1, 13] and stats[1, 1].tolist() == [2, 1]


def test_absent_class_gives_zero_statistics():
    m = np.ones((2, 3, 3), np.int64)
    for method, conn in CONNECTIVITIES:
        labels, stats, largest = OC.components(m, 4, method, conn)
        assert np.all(stats[:, [0, 2, 3]] == 0)
        assert np.all(stats[:, 1] == [1, 9 if method == "2d" else 18])
        assert np.array_equal(largest, m)
        assert np.all(labels[0] == 0) and np.all(labels[1] == (9 if method == "2d" else 0))


@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 1, 17), (17, 1, 1)])
def test_degenerate_grids(shape):
    rng = np.random.default_rng(3)
    m = OH.salt_pepper(rng, shape, 2)
    for method, conn in CONNECTIVITIES:
        got = OC.components(m, 2, method, conn)
        assert_same(got, OC.components_bfs(m, 2, method, conn))
        if shape[0] > 1 and method == "2d":   # every slice is one pixel: one component each
            assert np.all(got[1].sum(1)[:, 0] == 1) and np.array_equal(got[0].ravel(), np.arange(m.size))


def test_connectivity_counts_on_a_checkerboard():
    z, y, x = np.indices((4, 6, 6))
    m = ((z + y + x) % 2).astype(np.int64)
    assert OC.components(m, 2, "2d", 1)[1][:, :, 0].tolist() == [[18, 18]] * 4
    assert OC.components(m, 2, "2d", 2)[1][:, :, 0].tolist() == [[1, 1]] * 4
    assert OC.components(m, 2, "3d", 1)[1][0, :, 0].tolist() == [72, 72]
    assert OC.components(m, 2, "3d", 2)[1][0, :, 0].tolist() == [1, 1]
