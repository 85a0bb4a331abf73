"""CPU: the Hausdorff oracle (oracle/oracle_hausdorff.py, scipy restatement of medpy.metric.binary.hd) against the brute
force over border coordinates, and the C ABI's argument checks of the Hausdorff entry points (nothing launched)."""
import ctypes

import numpy as np
import pytest

import oracle_hausdorff as OH

SPACINGS_2D = [None, (1.0, 1.0), (1.5625, 0.7), (3.0, 0.25)]
SPACINGS_3D = [None, (1.0, 1.0, 1.0), (10.0, 1.5625, 1.5625), (0.5, 2.0, 1.25)]


def _check(pred, gt, C, method, spacing):
    a = OH.hausdorff(pred, gt, C, method, spacing)
    b = OH.hausdorff(pred, gt, C, method, spacing, brute=True)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    np.testing.assert_allclose(a[~np.isnan(a)], b[~np.isnan(b)], rtol=1e-12, atol=0)
    return a


@pytest.mark.parametrize("spacing", SPACINGS_2D)
@pytest.mark.parametrize("shape,C", [((3, 17, 23), 3), ((2, 32, 32), 4), ((2, 9, 40), 2)])
def test_oracle_2d_matches_brute_force(shape, C, spacing):
    rng = np.random.default_rng(hash((shape, C)) % 2**32)
    for maker in (OH.blobs, lambda r, s, c: OH.salt_pepper(r, s, c)):
        pred, gt = maker(rng, shape, C), maker(rng, shape, C)
        _check(pred, gt, C, "2d", spacing)


@pytest.mark.parametrize("spacing", SPACINGS_3D)
@pytest.mark.parametrize("shape,C", [((5, 13, 11), 3), ((4, 16, 16), 4)])
def test_oracle_3d_matches_brute_force(shape, C, spacing):
    rng = np.random.default_rng(7 + shape[0])
    pred, gt = OH.blobs(rng, shape, C), OH.blobs(rng, shape, C)
    _check(pred, gt, C, "3d", spacing)
    _check(OH.salt_pepper(rng, shape, C), gt, C, "3d", spacing)


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_oracle_empty_sets_are_nan(method):
    pred = np.zeros((2, 6, 7), np.int64)
    gt = np.zeros((2, 6, 7), np.int64)
    gt[:, 2:4, 3] = 1
    pred[:, 1, 1] = 2
    a = _check(pred, gt, 4, method, None)
    assert not np.isnan(a[:, 0]).any()           # class 0 present on both sides
    assert np.isnan(a[:, 1]).all()               # empty pred
    assert np.isnan(a[:, 2]).all()               # empty gt
    assert np.isnan(a[:, 3]).all()               # both empty


def test_oracle_edge_cases():
    # single pixels: the distance between them
    p = np.zeros((1, 9, 9), np.int64); g = np.zeros((1, 9, 9), np.int64)
    p[0, 1, 2] = 1; g[0, 7, 5] = 1
    a = _check(p, g, 2, "2d", (2.0, 0.5))
    assert a[0, 1] == pytest.approx(np.hypot(6 * 2.0, 3 * 0.5), rel=1e-15)
    # a class covering the whole grid: its border is the frame
    full = np.ones((1, 8, 10), np.int64)
    g = full.copy(); g[0, 3:5, 4:6] = 0
    a = _check(full, g, 2, "2d", None)
    assert np.isnan(a[0, 0]) and np.isfinite(a[0, 1])
    # masks touching the frame, identical maps, lines of one row / one column
    rng = np.random.default_rng(3)
    for shape in [(2, 1, 31), (2, 29, 1), (1, 1, 1), (3, 12, 12)]:
        m = OH.blobs(rng, shape, 3, smooth=1.5) if min(shape[1:]) > 1 else OH.salt_pepper(rng, shape, 3)
        for method in ("2d", "3d"):
            a = _check(m, m, 3, method, None)
            assert np.all((a == 0) | np.isnan(a))
            _check(m, OH.salt_pepper(rng, shape, 3), 3, method, (1.5, 0.5) if method == "2d" else (2.0, 1.5, 0.5))


def test_hausdorff_abi_rejects_bad_arguments():
    """Argument checks run on the host before anything is launched (no GPU needed)."""
    import dct_b200
    h = dct_b200._lib.lib()
    assert h.dct_hausdorff_scratch_bytes(4, 10, 256, 256, 0) >= 10 * 256 * 256 * (4 * 4 + 2)
    assert h.dct_hausdorff_scratch_bytes(4, 10, 256, 256, 1) >= 10 * 256 * 256 * (12 * 4 + 2)
    assert h.dct_hausdorff_scratch_bytes(65, 1, 8, 8, 0) == 0
    assert h.dct_hausdorff_scratch_bytes(4, 1, 32769, 8, 0) == 0
    assert h.dct_hausdorff_scratch_bytes(4, 40000, 8, 8, 0) > 0     # B is no distance axis in '2d' ...
    assert h.dct_hausdorff_scratch_bytes(4, 40000, 8, 8, 1) == 0    # ... but it is in a volume
    fake = 1 << 20   # aligned non-null stand-ins: rejected before any dereference
    sp = (ctypes.c_double * 3)(1.0, -1.0, 1.0)
    assert h.dct_hausdorff_i64(fake, fake, 4, 2, 8, 8, 0, sp, fake, None, fake, None) == -1     # (sy, sx) = (1, -1)
    sp = (ctypes.c_double * 3)(1.0, 1.0, float("nan"))
    assert h.dct_hausdorff_i64(fake, fake, 4, 2, 8, 8, 1, sp, fake, None, fake, None) == -1
    sp = (ctypes.c_double * 3)(0.0, 1.0, 1.0)
    assert h.dct_hausdorff_i64(fake, fake, 4, 2, 8, 8, 1, sp, fake, None, fake, None) == -1
    assert h.dct_hausdorff_i64(fake, fake, 65, 2, 8, 8, 0, None, fake, None, fake, None) == -2
    assert h.dct_hausdorff_i64(fake, fake, 4, 2, 8, 32769, 0, None, fake, None, fake, None) == -2
    assert h.dct_hausdorff_i64(None, fake, 4, 2, 8, 8, 0, None, fake, None, fake, None) == -1
    assert h.dct_hausdorff_i64(fake, fake, 4, 2, 8, 8, 0, None, fake, None, None, None) == -1
    assert h.dct_hausdorff_i64(fake + 4, fake, 4, 2, 8, 8, 0, None, fake, None, fake, None) == -3
