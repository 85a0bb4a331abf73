"""CPU: the surface-distance oracle (oracle/oracle_surface.py, scipy restatement of medpy hd95 / asd / assd) against the
brute force over border coordinates, the scalar 95th-percentile formula the kernels use against ``np.percentile``, and the
C ABI's argument checks of the surface-distance entry points (nothing launched)."""
import ctypes

import numpy as np
import pytest

import oracle_hausdorff as OH
import oracle_surface as OS

SPACINGS_2D = [None, (1.5625, 0.7), (3.0, 0.25)]
SPACINGS_3D = [None, (10.0, 1.5625, 1.5625), (0.5, 2.0, 1.25)]


def _check(pred, gt, C, method, spacing):
    a = OS.surface(pred, gt, C, method, spacing)
    b = OS.surface(pred, gt, C, method, spacing, brute=True)
    for k in OS.KEYS:
        assert np.array_equal(np.isnan(a[k]), np.isnan(b[k])), k
        np.testing.assert_allclose(a[k][~np.isnan(a[k])], b[k][~np.isnan(b[k])], rtol=1e-12, atol=0, err_msg=k)
    np.testing.assert_array_equal(a["hd"], OH.hausdorff(pred, gt, C, method, spacing))
    return a


@pytest.mark.parametrize("spacing", SPACINGS_2D)
@pytest.mark.parametrize("shape,C", [((3, 17, 23), 3), ((2, 32, 32), 4), ((2, 9, 40), 2)])
def test_oracle_2d_matches_brute_force(shape, C, spacing):
    rng = np.random.default_rng(shape[1] * 100 + C)
    for maker in (OH.blobs, OH.salt_pepper):
        _check(maker(rng, shape, C), maker(rng, shape, C), C, "2d", spacing)


@pytest.mark.parametrize("spacing", SPACINGS_3D)
@pytest.mark.parametrize("shape,C", [((5, 13, 11), 3), ((4, 16, 16), 4)])
def test_oracle_3d_matches_brute_force(shape, C, spacing):
    rng = np.random.default_rng(17 + shape[0])
    pred, gt = OH.blobs(rng, shape, C), OH.blobs(rng, shape, C)
    _check(pred, gt, C, "3d", spacing)
    _check(OH.salt_pepper(rng, shape, C), gt, C, "3d", spacing)


def test_oracle_directions_and_empty_sets():
    rng = np.random.default_rng(5)
    p, g = OH.blobs(rng, (2, 20, 24), 3), OH.blobs(rng, (2, 20, 24), 3)
    g[1][g[1] == 2] = 0   # class 2 absent from one label slice
    a, b = _check(p, g, 3, "2d", (1.5, 0.5)), _check(g, p, 3, "2d", (1.5, 0.5))
    for k in ("hd", "hd95", "assd"):   # symmetric
        np.testing.assert_allclose(a[k], b[k], rtol=1e-15)
    assert np.isnan(a["asd"][1, 2]) and np.isnan(a["hd95"][1, 2]) and not np.isnan(a["asd"][0, 2])
    assert not np.allclose(a["asd"][0], b["asd"][0])   # directional
    one = np.zeros((1, 12, 12), np.int64); sq = one.copy()
    one[0, 1, 1] = 1; sq[0, 4:10, 4:10] = 1           # 1 + 20 border pixels: (n - 1) * 0.95 = 19 exactly
    r = _check(one, sq, 2, "2d", None)
    s_pg = OS.surface_distances(one[0] == 1, sq[0] == 1)
    s_gp = OS.surface_distances(sq[0] == 1, one[0] == 1)
    assert s_pg.size == 1 and s_gp.size == 20 and 20 * 0.95 == 19.0
    assert r["hd95"][0, 1] == np.sort(np.hstack((s_pg, s_gp)))[19]   # t == 0: the key at rank 19 itself


def _percentile_cases():
    rng = np.random.default_rng(2024)
    for n in range(1, 3001):
        kind = n % 3
        if kind == 0:
            x = rng.standard_normal(n) * 10
        elif kind == 1:
            x = np.sqrt(rng.integers(0, 40, n).astype(np.float64))   # ties, as distances on a grid give
        else:
            x = np.sqrt(rng.integers(0, 4000, n).astype(np.float64)) * 1.5625
        yield x
    for n in (20 * 100 + 1, 20 * 12345 + 1, 1_000_001, 2_000_000, 4_194_305):   # large n; (n - 1) * 0.95 integral for most
        yield np.sqrt(rng.integers(0, 1 << 20, n).astype(np.float64))


def test_percentile_formula_equals_numpy_bitwise():
    integral = 0
    for x in _percentile_cases():
        want = np.percentile(x, 95)
        got = OS.percentile95(x)
        assert np.float64(got).view(np.uint64) == np.float64(want).view(np.uint64), (x.size, got, want)
        v = (x.size - 1) * 0.95
        integral += v == np.floor(v)
    assert integral >= 100


def test_surface_abi_rejects_bad_arguments():
    """Argument checks run on the host before anything is launched (no GPU needed); same codes as dct_hausdorff_i64."""
    import dct_b200
    h = dct_b200._lib.lib()
    for shape in [(4, 10, 256, 256, 0), (4, 10, 256, 256, 1), (19, 3, 17, 23, 0), (2, 40000, 8, 8, 0)]:
        C, B, H, W, vol = shape
        hd = h.dct_hausdorff_scratch_bytes(*shape)
        sd = h.dct_surface_distance_scratch_bytes(*shape)
        lines = 2 * C * (H * W if vol else B * H)
        rows = 1 if vol else B
        assert sd >= hd + 8 * B * H * W + 12 * lines + 2112 * rows * C
        assert sd <= hd + 8 * B * H * W + 12 * lines + 2112 * rows * C + 5 * 256
    assert h.dct_surface_distance_scratch_bytes(65, 1, 8, 8, 0) == 0
    assert h.dct_surface_distance_scratch_bytes(4, 1, 32769, 8, 0) == 0
    assert h.dct_surface_distance_scratch_bytes(4, 40000, 8, 8, 1) == 0
    assert h.dct_surface_distance_scratch_bytes(0, 1, 8, 8, 0) == 0
    fake = 1 << 20   # aligned non-null stand-ins: rejected before any dereference
    f = h.dct_surface_distances_i64
    sp = (ctypes.c_double * 3)(1.0, -1.0, 1.0)
    assert f(fake, fake, 4, 2, 8, 8, 0, sp, fake, None, fake, None) == -1
    sp = (ctypes.c_double * 3)(1.0, 1.0, float("nan"))
    assert f(fake, fake, 4, 2, 8, 8, 1, sp, fake, None, fake, None) == -1
    sp = (ctypes.c_double * 3)(0.0, 1.0, 1.0)
    assert f(fake, fake, 4, 2, 8, 8, 1, sp, fake, None, fake, None) == -1
    assert f(fake, fake, 65, 2, 8, 8, 0, None, fake, None, fake, None) == -2
    assert f(fake, fake, 4, 2, 8, 32769, 0, None, fake, None, fake, None) == -2
    assert f(None, fake, 4, 2, 8, 8, 0, None, fake, None, fake, None) == -1
    assert f(fake, fake, 4, 2, 8, 8, 0, None, None, None, fake, None) == -1
    assert f(fake, fake, 4, 2, 8, 8, 0, None, fake, None, None, None) == -1
    assert f(fake + 4, fake, 4, 2, 8, 8, 0, None, fake, None, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 0, None, fake + 2, None, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 0, None, fake, None, fake + 128, None) == -3
