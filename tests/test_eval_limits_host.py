"""CPU: the shape limits of the evaluation-path entry points (Hausdorff, surface distances, surface Dice, connected
components) at their boundaries, checked through the host-only scratch queries and through the entry points' argument
checks, which reject an unsupported shape before any CUDA call.

Limits (include/dct_b200.h): for the distance entry points H, W (and B of a volume) <= 32768, 2*C*B*max(H,W) <= 2^31 - 1
and, for a volume, 2*C*H*W <= 2^31 - 1; for the components B*H*W <= 2^31 - 1.  A scratch query returns 0 for a shape its
entry point rejects; otherwise it returns the size given by the header's per-pixel / per-line formulas."""
import ctypes

import pytest

INT_MAX = 2 ** 31 - 1
AXIS = 32768
DIST_QUERIES = ("dct_hausdorff_scratch_bytes", "dct_surface_distance_scratch_bytes", "dct_surface_dice_scratch_bytes")
ALL_QUERIES = DIST_QUERIES + ("dct_components_scratch_bytes",)


@pytest.fixture(scope="module")
def h():
    import dct_b200
    return dct_b200._lib.lib()


def a256(v):
    return (v + 255) // 256 * 256


def hd_layout(C, B, H, W, volume):
    """(hausdorff, surface distance, surface Dice) scratch bytes from the header's formulas, each region rounded up to
    256 bytes in the order the header lists them."""
    N, rows = B * H * W, 1 if volume else B
    fold_lines = 2 * C * (H * W if volume else B * H)   # lines of the last distance pass
    hd = a256(rows * C * 2 * 2 * 4)                     # per (row, class, side): maximum and presence words
    hd = a256(hd + N * 2)                               # per pixel: both maps' border records
    hd = a256(hd + 2 * C * N * 2)                       # per (side, class, pixel): column distance
    if volume:
        hd = a256(hd + 2 * C * N * 4)                   # per (side, class, pixel): d^2 after the row pass
    sd = a256(hd + 2 * N * 4)                           # per (side, pixel): d^2 of the queries
    sd = a256(sd + fold_lines * 8)                      # per line: sum of distances
    sd = a256(sd + fold_lines * 4)                      # per line: query count
    sd = a256(sd + rows * C * 256 * 8)                  # per (row, class): radix histogram
    sd = a256(sd + rows * C * 64)                       # per (row, class): select state
    nsd = a256(a256(hd + fold_lines * 4) + fold_lines * 4)   # per line: queries, queries within the tolerance
    return hd, sd, nsd


def cc_layout(C, B, H, W, volume):
    N, nrc = B * H * W, (1 if volume else B) * C
    return a256(a256(a256(a256(a256(N) + 4 * N) + 4 * N) + 8 * nrc) + 8 * nrc)


def sizes(h, C, B, H, W, volume):
    return [getattr(h, q)(C, B, H, W, volume) for q in ALL_QUERIES]


def assert_accepted(h, C, B, H, W, volume, queries=ALL_QUERIES):
    for q in queries:
        assert getattr(h, q)(C, B, H, W, volume) > 0, (q, C, B, H, W, volume)


def assert_rejected(h, C, B, H, W, volume, queries=ALL_QUERIES):
    for q in queries:
        assert getattr(h, q)(C, B, H, W, volume) == 0, (q, C, B, H, W, volume)


@pytest.mark.parametrize("volume", [0, 1])
def test_axis_length_boundary(h, volume):
    for C in (1, 2, 64):
        assert_accepted(h, C, 1, AXIS, 1, volume, DIST_QUERIES)
        assert_accepted(h, C, 1, 1, AXIS, volume, DIST_QUERIES)
        assert_rejected(h, C, 1, AXIS + 1, 1, volume, DIST_QUERIES)
        assert_rejected(h, C, 1, 1, AXIS + 1, volume, DIST_QUERIES)
        # the components have no axis limit of their own
        assert_accepted(h, C, 1, AXIS + 1, 1, volume, ALL_QUERIES[3:])
        assert_accepted(h, C, 1, 1, AXIS + 1, volume, ALL_QUERIES[3:])
    assert_accepted(h, 3, AXIS, 1, 1, volume, DIST_QUERIES)
    if volume:
        assert_rejected(h, 3, AXIS + 1, 1, 1, volume, DIST_QUERIES)
    else:
        assert_accepted(h, 3, 4 * AXIS, 1, 1, volume, DIST_QUERIES)   # slices: B is no axis of a grid


@pytest.mark.parametrize("volume", [0, 1])
def test_line_count_boundary(h, volume):
    """2*C*B*max(H,W) <= 2^31 - 1: 2*64*511*32768 = 2^31 - 2^24 is accepted, B = 512 (2^31) is not; and 2^31 - 2 =
    2*33*3171*10261 (2^30 - 1 = 3^2*7*11*31*151*331) is accepted, one more column or row is not."""
    assert 2 * 64 * 511 * AXIS <= INT_MAX < 2 * 64 * 512 * AXIS
    assert 2 * 33 * 3171 * 10261 == INT_MAX - 1
    for H, W in ((1, AXIS), (AXIS, 1), (AXIS, 7)):
        assert_accepted(h, 64, 511, H, W, volume, DIST_QUERIES)
        assert_rejected(h, 64, 512, H, W, volume, DIST_QUERIES)
    for H, W in ((1, 10261), (10261, 1), (10261, 3)):
        assert_accepted(h, 33, 3171, H, W, volume, DIST_QUERIES)
        assert_rejected(h, 33, 3171, H + (H >= W), W + (W > H), volume, DIST_QUERIES)
        assert_rejected(h, 33, 3172, H, W, volume, DIST_QUERIES)
        assert_rejected(h, 34, 3171, H, W, volume, DIST_QUERIES)


def test_volume_plane_boundary(h):
    """A volume also needs 2*C*H*W <= 2^31 - 1 (the lines of its last pass): 2*33*10261*3171 = 2^31 - 2 is accepted, one
    more column is not; the same slice batch has no such limit."""
    assert_accepted(h, 33, 1, 10261, 3171, 1, DIST_QUERIES)
    assert_accepted(h, 33, 2, 3171, 10261, 1, DIST_QUERIES)
    assert_rejected(h, 33, 1, 10261, 3172, 1, DIST_QUERIES)
    assert_rejected(h, 33, 2, 3172, 10261, 1, DIST_QUERIES)
    assert_accepted(h, 33, 1, 10261, 3172, 0, DIST_QUERIES)
    assert_accepted(h, 33, 2, 3172, 10261, 0, DIST_QUERIES)


def test_distance_limits_do_not_overflow(h):
    """Shapes whose line count overflows int64 arithmetic are rejected, not wrapped into range."""
    for C, B in ((1, 2 ** 62), (64, 2 ** 56), (64, 2 ** 61), (1, 2 ** 63 - 1), (2, INT_MAX), (1, INT_MAX // 2 + 1)):
        for volume in (0, 1):
            assert_rejected(h, C, B, 1, 1, volume, DIST_QUERIES)
    assert_accepted(h, 1, INT_MAX // 2, 1, 1, 0, DIST_QUERIES)


@pytest.mark.parametrize("volume", [0, 1])
def test_component_pixel_boundary(h, volume):
    """B*H*W <= 2^31 - 1 (a prime: only 1 x 1 x (2^31 - 1) and its permutations reach it); B*H likewise; factors that
    would overflow int64 are rejected."""
    q = ALL_QUERIES[3:]
    for shape in ((1, 1, INT_MAX), (1, INT_MAX, 1), (INT_MAX, 1, 1), (1, 46340, 46341), (46341, 46340, 1)):
        assert_accepted(h, 2, *shape, volume, q)
    for shape in ((1, 1, INT_MAX + 1), (1, INT_MAX + 1, 1), (INT_MAX + 1, 1, 1), (2 ** 16, 2 ** 15, 1),
                  (1, 2 ** 16, 2 ** 15), (2, 2 ** 15, 2 ** 15), (1, 46341, 46341), (2 ** 40, 2 ** 40, 2 ** 40),
                  (2 ** 62, 2 ** 62, 1)):
        assert_rejected(h, 2, *shape, volume, q)
    assert_accepted(h, 64, 1, 1, INT_MAX, volume, q)
    assert_rejected(h, 65, 1, 1, 1, volume, q)


def test_classes_and_positive_axes(h):
    for volume in (0, 1):
        assert_accepted(h, 64, 2, 3, 4, volume)
        assert_rejected(h, 65, 2, 3, 4, volume)
        for bad in ((0, 2, 3, 4), (2, 0, 3, 4), (2, 2, 0, 4), (2, 2, 3, 0), (-1, 2, 3, 4), (2, -1, 3, 4)):
            assert_rejected(h, *bad, volume)


@pytest.mark.parametrize("volume", [0, 1])
def test_scratch_sizes_follow_the_header_formulas(h, volume):
    shapes = [(1, 1, 1, 1), (2, 3, 17, 23), (19, 5, 33, 47), (4, 10, 256, 256), (2, 8, 512, 512), (64, 7, 1, 1),
              (3, 2, 48, 16384), (4, 1, 32768, 24), (3, 16384, 6, 5), (3, 32768, 2, 3), (64, 511, 1, AXIS),
              (33, 3171, 10261, 1), (33, 1, 10261, 3171)]
    for C, B, H, W in shapes:
        got = sizes(h, C, B, H, W, volume)
        want = list(hd_layout(C, B, H, W, volume)) + [cc_layout(C, B, H, W, volume)]
        assert got == want, (C, B, H, W, volume)
        assert all(v % 256 == 0 for v in got)
    for C, B, H, W in ((2, 1, 46340, 46341), (2, 1, 1, INT_MAX), (2, INT_MAX, 1, 1)):
        assert h.dct_components_scratch_bytes(C, B, H, W, volume) == cc_layout(C, B, H, W, volume)


def _ptr(v=4096):
    return ctypes.c_void_p(v)


def test_entry_points_reject_unsupported_shapes_before_any_launch(h):
    """Non-null, aligned dummy pointers and a rejected shape: DCT_ERR_UNSUPPORTED, decided on the host before any CUDA call
    (no device is needed, and a dereference of the dummy pointers would fault)."""
    import dct_b200
    UNSUP = dct_b200._lib.ERR_UNSUPPORTED
    tol = (ctypes.c_double * 65)(*([1.0] * 65))
    sp = (ctypes.c_double * 3)(1.0, 1.0, 1.0)
    rejected = [(2, 1, AXIS + 1, 1, 0), (2, 1, 1, AXIS + 1, 1), (2, AXIS + 1, 1, 1, 1), (64, 512, 1, AXIS, 0),
                (33, 3171, 10262, 1, 1), (33, 1, 10261, 3172, 1), (65, 1, 4, 4, 0), (64, 2 ** 61, 1, 1, 0)]
    p = _ptr()
    for C, B, H, W, volume in rejected:
        for spacing in (None, sp):
            assert h.dct_hausdorff_i64(p, p, C, B, H, W, volume, spacing, p, p, p, None) == UNSUP
            assert h.dct_surface_distances_i64(p, p, C, B, H, W, volume, spacing, p, p, p, None) == UNSUP
            assert h.dct_surface_dice_i64(p, p, C, B, H, W, volume, spacing, tol, p, p, p, p, None) == UNSUP
    for C, B, H, W in ((2, 1, 1, INT_MAX + 1), (2, 2 ** 16, 2 ** 15, 1), (2, 1, 46341, 46341), (65, 1, 4, 4),
                       (2, 2 ** 40, 2 ** 40, 2 ** 40)):
        for volume, conn in ((0, 1), (0, 2), (1, 1), (1, 3)):
            assert h.dct_components_i64(p, C, B, H, W, volume, conn, p, p, _ptr(8192), p, p, None) == UNSUP
