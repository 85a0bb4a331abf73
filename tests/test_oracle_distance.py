"""CPU: the distance map oracle (oracle/oracle_distance.py) against its brute force, hand cases of the definition, and the
C ABI's scratch query, limits and argument checks of dct_distance_map_i64 (nothing launched)."""
import ctypes

import numpy as np
import pytest
from scipy.ndimage import distance_transform_edt

import oracle_distance as ODM
import oracle_hausdorff as OH

SPACINGS_2D = [None, (1.5625, 0.7), (3.0, 0.25)]
SPACINGS_3D = [None, (10.0, 1.5625, 1.5625), (0.5, 2.0, 1.25)]
INT_MAX = 2 ** 31 - 1
AXIS = 32768


def _check(m, C, first, method, spacing, signed):
    a = ODM.distance_map(m, C, first, method, spacing, signed)
    b = ODM.distance_map(m, C, first, method, spacing, signed, brute=True)
    assert a.shape == (m.shape[0], C - first) + m.shape[1:]
    if spacing is None:   # unit spacing: both are the square root of the same integer
        np.testing.assert_array_equal(a, b)
    else:
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=0)
    return a


@pytest.mark.parametrize("signed", [True, False])
@pytest.mark.parametrize("spacing", SPACINGS_2D)
@pytest.mark.parametrize("shape,C", [((3, 17, 23), 3), ((2, 32, 32), 4), ((2, 9, 40), 2)])
def test_oracle_2d_matches_brute_force(shape, C, spacing, signed):
    rng = np.random.default_rng(shape[1] * 100 + C)
    for maker in (OH.blobs, OH.salt_pepper):
        m = maker(rng, shape, C)
        for first in (0, 1):
            _check(m, C, first, "2d", spacing, signed)


@pytest.mark.parametrize("signed", [True, False])
@pytest.mark.parametrize("spacing", SPACINGS_3D)
@pytest.mark.parametrize("shape,C", [((5, 13, 11), 3), ((4, 16, 16), 4)])
def test_oracle_3d_matches_brute_force(shape, C, spacing, signed):
    rng = np.random.default_rng(17 + shape[0])
    for maker in (OH.blobs, OH.salt_pepper):
        _check(maker(rng, shape, C), C, 0, "3d", spacing, signed)


def test_binary_inside_map_is_scipy():
    rng = np.random.default_rng(5)
    m = OH.blobs(rng, (3, 30, 26), 2)
    for sp in SPACINGS_2D:
        got = ODM.distance_map(m, 2, 1, "2d", sp, signed=False)[:, 0]
        for b in range(3):
            np.testing.assert_array_equal(got[b], distance_transform_edt(m[b] != 0, sampling=sp))


def test_absent_and_filling_classes():
    m = np.zeros((2, 5, 6), np.int64)
    m[1, 2, 3] = 1
    s = _check(m, 3, 0, "2d", None, True)
    assert np.all(s[0] == 0.0)                     # slice 0: class 0 fills it, classes 1 and 2 are absent
    assert np.all(s[1, 2] == 0.0)                  # class 2 absent from slice 1
    assert s[1, 1, 2, 3] == -1.0 and s[1, 1, 0, 0] == np.sqrt(13.0)
    assert s[1, 0, 2, 3] == 1.0 and s[1, 0, 2, 4] == -1.0
    d = _check(m, 3, 0, "2d", None, False)
    assert np.all(np.isinf(d[0, 0])) and np.all(d[0, 1:] == 0.0)
    assert d[1, 0, 2, 3] == 0.0 and d[1, 1, 2, 3] == 1.0 and d[1, 1].sum() == 1.0
    # scipy's artifact on a grid without background, which the oracle replaces by +inf
    assert not np.all(np.isinf(distance_transform_edt(np.ones((3, 4), bool))))
    v = _check(m, 3, 0, "3d", None, True)
    assert np.all(v[:, 2] == 0.0) and v[1, 1, 2, 3] == -1.0 and v[0, 1, 2, 3] == 1.0


def test_out_of_range_values_are_outside_every_class():
    m = np.zeros((1, 4, 5), np.int64)
    m[0, 1, 1] = 7; m[0, 2, 3] = -1
    s = _check(m, 2, 0, "2d", None, True)
    assert s[0, 0, 1, 1] == 1.0 and s[0, 0, 2, 3] == 1.0      # outside class 0, next to it
    assert np.all(s[0, 1] == 0.0)                              # class 1 absent: its plane is 0
    d = _check(m, 2, 0, "2d", None, False)
    assert d[0, 0, 1, 1] == 0.0 and d[0, 0, 1, 2] == 1.0


@pytest.mark.parametrize("method", ["2d", "3d"])
def test_degenerate_grids(method):
    rng = np.random.default_rng(2)
    for shape in [(1, 1, 1), (1, 1, 37), (29, 1, 1), (3, 1, 19)]:
        for maker in (OH.salt_pepper, lambda r, s, c: np.zeros(s, np.int64)):
            m = maker(rng, shape, 3)
            for signed in (True, False):
                _check(m, 3, 0, method, None, signed)
                _check(m, 3, 1, method, (2.0, 0.5, 0.75)[3 - (2 if method == "2d" else 3):], signed)
    one = ODM.distance_map(np.ones((1, 1, 1), np.int64), 2, 1, method, None, signed=False)
    assert one.shape == (1, 1, 1, 1) and np.isinf(one[0, 0, 0, 0])
    assert np.all(ODM.distance_map(np.ones((1, 1, 1), np.int64), 2, 0, method, None) == 0.0)


@pytest.fixture(scope="module")
def h():
    import dct_b200
    return dct_b200._lib.lib()


def a256(v):
    return (v + 255) // 256 * 256


def layout(C, first, B, H, W, volume, signed):
    """The header's formula: 8 per (row, computed class), 1 per pixel, 2*S*Cc per pixel, and for a volume 4*S*Cc per
    pixel, each region rounded up to 256 bytes."""
    Cc, N, S = C - first, B * H * W, 2 if signed else 1
    v = a256(a256(a256((1 if volume else B) * Cc * 8) + N) + 2 * S * Cc * N)
    return a256(v + 4 * S * Cc * N) if volume else v


@pytest.mark.parametrize("volume", [0, 1])
def test_scratch_sizes_follow_the_header_formula(h, volume):
    shapes = [(1, 1, 1, 1), (2, 3, 17, 23), (19, 5, 33, 47), (4, 10, 256, 256), (2, 8, 512, 512), (64, 7, 1, 1),
              (3, 2, 48, 16384), (4, 1, 32768, 24), (3, 16384, 6, 5)]
    for C, B, H, W in shapes:
        for first in sorted({0, 1, C - 1}):
            if first >= C:
                continue
            for signed in (0, 1):
                got = h.dct_distance_map_scratch_bytes(C, first, B, H, W, volume, signed)
                assert got == layout(C, first, B, H, W, volume, signed), (C, first, B, H, W, volume, signed)
                assert got % 256 == 0


def _ok(h, C, first, B, H, W, volume):
    return all(h.dct_distance_map_scratch_bytes(C, first, B, H, W, volume, s) > 0 for s in (0, 1))


def _rejected(h, C, first, B, H, W, volume):
    return all(h.dct_distance_map_scratch_bytes(C, first, B, H, W, volume, s) == 0 for s in (0, 1))


@pytest.mark.parametrize("volume", [0, 1])
def test_limits_at_their_boundaries(h, volume):
    """The Hausdorff limits applied to the computed class count C - first_class, and C <= 64."""
    for C, first in ((1, 0), (2, 1), (64, 0), (64, 63)):
        assert _ok(h, C, first, 1, AXIS, 1, volume) and _ok(h, C, first, 1, 1, AXIS, volume)
        assert _rejected(h, C, first, 1, AXIS + 1, 1, volume) and _rejected(h, C, first, 1, 1, AXIS + 1, volume)
    assert _ok(h, 3, 0, AXIS, 1, 1, volume)
    assert _rejected(h, 3, 0, AXIS + 1, 1, 1, volume) == bool(volume)
    # 2 * Cc * B * max(H, W) <= 2^31 - 1, with Cc = C - first_class
    assert _ok(h, 64, 0, 511, 1, AXIS, volume) and _rejected(h, 64, 0, 512, 1, AXIS, volume)
    assert _ok(h, 64, 32, 1023, 1, AXIS, volume) and _rejected(h, 64, 32, 1024, 1, AXIS, volume)
    assert _ok(h, 33, 0, 3171, 10261, 1, volume) and _rejected(h, 33, 0, 3172, 10261, 1, volume)
    assert _ok(h, 34, 1, 3171, 10261, 1, volume) and _rejected(h, 34, 1, 3171, 10262, 1, volume)
    assert _rejected(h, 65, 1, 1, 4, 4, volume) and _rejected(h, 65, 60, 1, 4, 4, volume)
    for C, B in ((1, 2 ** 62), (64, 2 ** 61), (2, INT_MAX)):
        assert _rejected(h, C, 0, B, 1, 1, volume)


def test_volume_plane_boundary(h):
    assert _ok(h, 33, 0, 1, 10261, 3171, 1) and _rejected(h, 33, 0, 1, 10261, 3172, 1)
    assert _ok(h, 33, 0, 1, 10261, 3172, 0)


def test_bad_arguments_give_no_size(h):
    for C, first, signed in ((2, 2, 1), (2, -1, 1), (0, 0, 1), (-1, 0, 0), (3, 1, 2), (3, 1, -1)):
        assert h.dct_distance_map_scratch_bytes(C, first, 1, 4, 4, 0, signed) == 0, (C, first, signed)
    for bad in ((0, 4, 4), (2, 0, 4), (2, 4, 0), (-1, 4, 4)):
        assert h.dct_distance_map_scratch_bytes(2, 0, *bad, 0, 1) == 0


def test_entry_point_rejects_before_any_launch(h):
    """Aligned non-null stand-ins that would fault if dereferenced: every rejection is decided on the host."""
    p = ctypes.c_void_p(1 << 20)
    f = h.dct_distance_map_i64

    def sp(*v):
        return (ctypes.c_double * len(v))(*v)

    def call(m=p, C=4, first=0, B=2, H=8, W=8, volume=0, spacing=None, signed=1, out=p, flags=None, scratch=p):
        return f(m, C, first, B, H, W, volume, spacing, signed, out, flags, scratch, None)

    for kw in (dict(first=4), dict(first=-1), dict(C=0), dict(signed=2), dict(signed=-1), dict(m=None),
               dict(out=None), dict(scratch=None), dict(B=0), dict(H=-1), dict(W=0),
               dict(spacing=sp(1.0, -1.0)), dict(spacing=sp(0.0, 1.0)), dict(spacing=sp(float("nan"), 1.0)),
               dict(spacing=sp(1.0, float("inf"))), dict(volume=1, spacing=sp(1.0, 1.0, -2.0)),
               dict(volume=1, spacing=sp(float("inf"), 1.0, 1.0))):
        assert call(**kw) == -1, kw
    for kw in (dict(C=65), dict(C=65, first=60), dict(H=AXIS + 1), dict(W=AXIS + 1), dict(volume=1, B=AXIS + 1),
               dict(C=64, B=512, H=1, W=AXIS), dict(volume=1, C=33, B=1, H=10261, W=3172)):
        for signed in (0, 1):
            assert call(signed=signed, **kw) == -2, kw
    assert call(m=ctypes.c_void_p((1 << 20) + 4)) == -3
    assert call(out=ctypes.c_void_p((1 << 20) + 2)) == -3
    assert call(flags=ctypes.c_void_p((1 << 20) + 2)) == -3
    assert call(scratch=ctypes.c_void_p((1 << 20) + 128)) == -3


def test_spacing_argument_parsing():
    import dct_b200
    sp = dct_b200.distance._spacing
    assert sp(None, "2d", "t") is None
    assert list(sp(2.0, "2d", "t")) == [2.0, 2.0] and list(sp(3, "3d", "t")) == [3.0, 3.0, 3.0]
    assert list(sp((10.0, 1.5, 1.25), "3d", "t")) == [10.0, 1.5, 1.25]
    with pytest.raises(AssertionError):
        sp((1.0, 2.0), "3d", "t")
