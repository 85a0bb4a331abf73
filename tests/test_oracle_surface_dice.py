"""CPU: the normalized surface Dice oracle (oracle/oracle_surface_dice.py) against its brute force over border coordinates,
hand cases of the definition, and the C ABI's scratch query and argument checks of dct_surface_dice_i64 (nothing
launched)."""
import ctypes
import math

import numpy as np
import pytest

import oracle_hausdorff as OH
import oracle_surface_dice as OD

SPACINGS_2D = [None, (1.5625, 0.7), (3.0, 0.25)]
SPACINGS_3D = [None, (10.0, 1.5625, 1.5625), (0.5, 2.0, 1.25)]
UNIT_TOLS = [0.0, 1.0, math.sqrt(2), 2.0, 3.5, math.sqrt(5)]


def _check(pred, gt, C, tol, method, spacing):
    if spacing is not None and tol > 0:   # EDT and cdist may round a distance differently in the last bit
        for per_class in OD.distances(pred, gt, C, method, spacing):
            for s_pg, s_gp in per_class:
                d = np.hstack((s_pg, s_gp))
                assert not np.any(np.abs(d - tol) <= 1e-9 * tol), f"tolerance {tol} is an attained distance"
    a = OD.surface_dice(pred, gt, C, tol, method, spacing)
    b = OD.surface_dice(pred, gt, C, tol, method, spacing, brute=True)
    assert a["counts"].dtype == np.int64 and a["counts"].shape == (1 if method == "3d" else pred.shape[0], C, 4)
    np.testing.assert_array_equal(a["counts"], b["counts"])
    for k in OD.KEYS:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    return a


def _tols(spacing):
    # unit spacing: attained distances included (inclusive comparison); otherwise values with no distance near them
    return UNIT_TOLS if spacing is None else [0.0, 1.2345, 2.8765, 7.6543]


@pytest.mark.parametrize("spacing", SPACINGS_2D)
@pytest.mark.parametrize("shape,C", [((3, 17, 23), 3), ((2, 32, 32), 4), ((2, 9, 40), 2)])
def test_oracle_2d_matches_brute_force(shape, C, spacing):
    rng = np.random.default_rng(shape[1] * 100 + C)
    for maker in (OH.blobs, OH.salt_pepper):
        p, g = maker(rng, shape, C), maker(rng, shape, C)
        for tol in _tols(spacing):
            _check(p, g, C, tol, "2d", spacing)


@pytest.mark.parametrize("spacing", SPACINGS_3D)
@pytest.mark.parametrize("shape,C", [((5, 13, 11), 3), ((4, 16, 16), 4)])
def test_oracle_3d_matches_brute_force(shape, C, spacing):
    rng = np.random.default_rng(17 + shape[0])
    p, g = OH.blobs(rng, shape, C), OH.blobs(rng, shape, C)
    for tol in _tols(spacing):
        _check(p, g, C, tol, "3d", spacing)
        _check(OH.salt_pepper(rng, shape, C), g, C, tol, "3d", spacing)


def test_per_class_tolerances_equal_single_class_calls():
    rng = np.random.default_rng(3)
    p, g = OH.blobs(rng, (2, 30, 28), 3), OH.blobs(rng, (2, 30, 28), 3)
    tols = [0.0, math.sqrt(2), 4.0]
    r = _check(p, g, 3, tols, "2d", None)
    for c, t in enumerate(tols):
        np.testing.assert_array_equal(r["counts"][:, c], OD.surface_dice(p, g, 3, t)["counts"][:, c])


def test_both_borders_empty_is_nan():
    p = np.zeros((1, 6, 7), np.int64); g = np.zeros((1, 6, 7), np.int64)
    r = _check(p, g, 2, 1.0, "2d", None)
    assert r["counts"][0, 1].tolist() == [0, 0, 0, 0]
    assert all(np.isnan(r[k][0, 1]) for k in OD.KEYS)
    assert r["nsd"][0, 0] == 1.0   # class 0 fills both grids: identical borders


def test_one_side_empty_scores_zero():
    p = np.zeros((2, 8, 9), np.int64); g = np.zeros((2, 8, 9), np.int64)
    g[0, 2:5, 3:6] = 1           # missed structure: prediction border empty
    p[1, 1:3, 1:3] = 1           # hallucinated structure: label border empty
    r = _check(p, g, 2, 100.0, "2d", None)
    assert r["counts"][0, 1].tolist() == [0, 0, 0, 8] and r["nsd"][0, 1] == 0.0
    assert np.isnan(r["overlap_pg"][0, 1]) and r["overlap_gp"][0, 1] == 0.0
    assert r["counts"][1, 1].tolist() == [0, 4, 0, 0] and r["nsd"][1, 1] == 0.0
    assert r["overlap_pg"][1, 1] == 0.0 and np.isnan(r["overlap_gp"][1, 1])


def test_identical_maps_score_one():
    rng = np.random.default_rng(7)
    for method in ("2d", "3d"):
        m = OH.blobs(rng, (3, 24, 20), 4)
        r = _check(m, m.copy(), 4, 0.0, method, None)
        present = r["counts"][..., 1] > 0
        assert present.any()
        assert np.all(r["nsd"][present] == 1.0) and np.all(r["overlap_pg"][present] == 1.0)
        np.testing.assert_array_equal(r["counts"][..., 0], r["counts"][..., 1])


def test_zero_tolerance_counts_coinciding_border_pixels():
    rng = np.random.default_rng(9)
    p, g = OH.salt_pepper(rng, (2, 15, 17), 3), OH.salt_pepper(rng, (2, 15, 17), 3)
    r = _check(p, g, 3, 0.0, "2d", None)
    for b in range(2):
        for c in range(3):
            bp, bg = OH.border(p[b] == c), OH.border(g[b] == c)
            assert r["counts"][b, c].tolist() == [int((bp & bg).sum()), int(bp.sum()), int((bp & bg).sum()),
                                                  int(bg.sum())]


def test_attained_tolerance_is_inclusive():
    # one prediction pixel at offsets (1, 2) from a one-pixel label: distance sqrt(5) at unit spacing
    p = np.zeros((1, 9, 9), np.int64); g = np.zeros((1, 9, 9), np.int64)
    p[0, 3, 3] = 1; g[0, 4, 5] = 1
    for tol, within in ((math.sqrt(5), 1), (np.nextafter(math.sqrt(5), 0), 0), (2.0, 0), (3.0, 1)):
        r = _check(p, g, 2, tol, "2d", None)
        assert r["counts"][0, 1].tolist() == [within, 1, within, 1], tol
    # anisotropic: (1 * 1.5, 2 * 0.5) -> sqrt(1.5^2 + 1) attained, inclusive
    sp = (1.5, 0.5)
    d = math.sqrt(1.5 ** 2 + 1.0)
    assert OD.surface_dice(p, g, 2, d, "2d", sp)["counts"][0, 1].tolist() == [1, 1, 1, 1]


def test_distances_helper_matches_counts():
    rng = np.random.default_rng(21)
    p, g = OH.blobs(rng, (2, 20, 22), 3), OH.blobs(rng, (2, 20, 22), 3)
    g[1][g[1] == 2] = 0
    r = OD.surface_dice(p, g, 3, 2.5, "2d", (1.5, 0.5))
    for row, per_class in enumerate(OD.distances(p, g, 3, "2d", (1.5, 0.5))):
        for c, (s_pg, s_gp) in enumerate(per_class):
            assert r["counts"][row, c].tolist() == [int((s_pg <= 2.5).sum()), s_pg.size, int((s_gp <= 2.5).sum()),
                                                    s_gp.size]


def test_surface_dice_scratch_bytes_and_limits():
    import dct_b200
    h = dct_b200._lib.lib()
    for shape in [(4, 10, 256, 256, 0), (4, 10, 256, 256, 1), (19, 3, 17, 23, 0), (2, 40000, 8, 8, 0)]:
        C, B, H, W, vol = shape
        hd = h.dct_hausdorff_scratch_bytes(*shape)
        nsd = h.dct_surface_dice_scratch_bytes(*shape)
        lines = 2 * C * (H * W if vol else B * H)
        assert hd + 8 * lines <= nsd <= hd + 8 * lines + 2 * 256
        assert nsd % 256 == 0
    assert h.dct_surface_dice_scratch_bytes(65, 1, 8, 8, 0) == 0
    assert h.dct_surface_dice_scratch_bytes(4, 1, 32769, 8, 0) == 0
    assert h.dct_surface_dice_scratch_bytes(4, 40000, 8, 8, 1) == 0
    assert h.dct_surface_dice_scratch_bytes(0, 1, 8, 8, 0) == 0


def test_surface_dice_abi_rejects_bad_arguments():
    """Argument checks run on the host before anything is launched (no GPU needed); codes as dct_hausdorff_i64."""
    import dct_b200
    h = dct_b200._lib.lib()
    fake = 1 << 20   # aligned non-null stand-ins: rejected before any dereference
    f = h.dct_surface_dice_i64

    def tol(*v):
        return (ctypes.c_double * len(v))(*v)

    ok = tol(1.0, 2.0, 0.0, 3.5)
    for bad in (tol(1.0, -1.0, 1.0, 1.0), tol(1.0, 1.0, float("nan"), 1.0), tol(float("inf"), 1.0, 1.0, 1.0),
                tol(1.0, 1.0, 1.0, -0.5), None):
        assert f(fake, fake, 4, 2, 8, 8, 0, None, bad, fake, None, None, fake, None) == -1
        assert f(fake, fake, 4, 2, 8, 8, 1, None, bad, fake, fake, None, fake, None) == -1
    for sp in (tol(1.0, -1.0, 1.0), tol(1.0, 1.0, float("nan")), tol(0.0, 1.0, 1.0), tol(1.0, float("inf"), 1.0)):
        assert f(fake, fake, 4, 2, 8, 8, 1, sp, ok, fake, None, None, fake, None) == -1
    assert f(fake, fake, 4, 2, 8, 8, 0, tol(1.0, 0.0), ok, fake, None, None, fake, None) == -1
    assert f(fake, fake, 65, 2, 8, 8, 0, None, ok, fake, None, None, fake, None) == -2
    assert f(fake, fake, 4, 2, 8, 32769, 0, None, ok, fake, None, None, fake, None) == -2
    assert f(None, fake, 4, 2, 8, 8, 0, None, ok, fake, None, None, fake, None) == -1
    assert f(fake, None, 4, 2, 8, 8, 0, None, ok, fake, None, None, fake, None) == -1
    assert f(fake, fake, 4, 2, 8, 8, 0, None, ok, None, None, None, fake, None) == -1
    assert f(fake, fake, 4, 2, 8, 8, 0, None, ok, fake, None, None, None, None) == -1
    assert f(fake + 4, fake, 4, 2, 8, 8, 0, None, ok, fake, None, None, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 0, None, ok, fake + 2, None, None, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 0, None, ok, fake, fake + 4, None, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 0, None, ok, fake, None, fake + 2, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 0, None, ok, fake, None, None, fake + 128, None) == -3


def test_tolerance_argument_parsing():
    import dct_b200
    tol = dct_b200.metrics._tolerances
    assert list(tol(1.5, 3)) == [1.5, 1.5, 1.5]
    assert list(tol([0, 1, math.sqrt(2)], 3)) == [0.0, 1.0, math.sqrt(2)]
    assert list(tol(np.array([2.0, 3.0]), 2)) == [2.0, 3.0]
    with pytest.raises(AssertionError):
        tol([1.0, 2.0], 3)
    for bad in (-1.0, float("nan"), float("inf"), [1.0, -0.1]):
        with pytest.raises(ValueError):
            tol(bad, 2)
