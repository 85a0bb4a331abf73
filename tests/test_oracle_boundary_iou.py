"""CPU: the Boundary IoU oracle (oracle/oracle_boundary_iou.py) -- the scipy restatement against the definition's own cv2
code and a brute-force window check --, hand cases of the definition, the band width rule, argument parsing, and the C
ABI's scratch query and argument checks of dct_boundary_iou_i64 (nothing launched)."""
import math

import numpy as np
import pytest
from scipy.ndimage import zoom

import oracle_boundary_iou as OB


def _random_maps(rng, n):
    """Blobs and salt-and-pepper maps with H or W from 1 to 39, C from 2 to 19, d from 1 past max(H, W)."""
    for t in range(n):
        H, W = (int(v) for v in rng.integers(1, 40, 2))
        if t % 5 == 0:
            H = 1
        elif t % 5 == 1:
            W = 1
        C = int(rng.integers(2, 20))
        d = int(rng.integers(1, max(H, W) + 3))
        if t % 2:
            M = rng.integers(0, C, (H, W))
        else:
            M = zoom(rng.integers(0, C, (H // 6 + 1, W // 6 + 1)), 7, order=0)[:H, :W]
        yield M, C, d


def test_scipy_restatement_equals_brute_force():
    rng = np.random.default_rng(0)
    for M, C, d in _random_maps(rng, 200):
        for c in range(C):
            np.testing.assert_array_equal(OB.mask_to_boundary(M == c, d), OB.mask_to_boundary_brute(M == c, d))


def test_scipy_restatement_equals_definition():
    pytest.importorskip("cv2")
    rng = np.random.default_rng(1)
    for M, C, d in _random_maps(rng, 300):
        for c in range(C):
            np.testing.assert_array_equal(OB.mask_to_boundary(M == c, d), OB.mask_to_boundary_cv2(M == c, d))


def test_full_class_is_a_ring_of_width_d():
    H, W, d = 20, 31, 4
    band = OB.mask_to_boundary(np.ones((H, W), bool), d)
    inner = np.zeros((H, W), bool)
    inner[d: H - d, d: W - d] = True
    np.testing.assert_array_equal(band, ~inner)
    assert band.sum() == H * W - (H - 2 * d) * (W - 2 * d)


def test_window_wider_than_the_image_makes_every_pixel_band():
    rng = np.random.default_rng(2)
    M = rng.integers(0, 3, (9, 30))
    for d in (5, 6, 40):   # 2d+1 > 9
        for c in range(3):
            np.testing.assert_array_equal(OB.mask_to_boundary(M == c, d), M == c)
    assert not np.array_equal(OB.mask_to_boundary(np.ones((9, 30), bool), 4), np.ones((9, 30), bool))


def test_identical_maps_score_one_and_absent_classes_nan():
    rng = np.random.default_rng(3)
    M = zoom(rng.integers(0, 3, (2, 5, 6)), (1, 8, 8), order=0)
    r = OB.boundary_iou(M, M.copy(), 5, 3)
    present = r["counts"][..., 1] > 0
    assert present[:, :3].any() and not present[:, 3:].any()
    assert np.all(r["biou"][present] == 1.0) and np.all(np.isnan(r["biou"][~present]))
    np.testing.assert_array_equal(r["counts"][..., 0], r["counts"][..., 1])
    np.testing.assert_array_equal(r["counts"][..., 0], r["counts"][..., 2])


def test_ignore_block_keeps_the_gt_band_and_leaves_every_count():
    C, d = 2, 2
    g = np.zeros((1, 12, 12), np.int64)
    g[0, :, 6:] = 255                  # right half ignored
    p = np.ones((1, 12, 12), np.int64)  # class 1 everywhere in the prediction
    r = OB.boundary_iou(p, g, C, d, ignore_index=255)
    band_g = OB.mask_to_boundary(g[0] == 0, d)
    assert band_g[:, 4:6].all()        # next to the ignore block: band of class 0
    I, G, P = r["counts"][0, 0]
    assert G == band_g.sum() and P == 0 and I == 0
    I, G, P = r["counts"][0, 1]        # class 1: band of P on the valid half only
    band_p = OB.mask_to_boundary(p[0] == 1, d)
    assert (I, G) == (0, 0) and P == (band_p & (g[0] != 255)).sum() == band_p[:, :6].sum()
    unmasked = OB.boundary_iou(p, np.where(g == 255, 0, g), C, d)   # the same label without the ignore region
    assert unmasked["counts"][0, 1, 2] > P


def test_ratio_is_the_double_quotient():
    assert OB.ratio((3, 5, 7)) == 3 / 9
    assert math.isnan(OB.ratio((0, 0, 0)))
    assert OB.ratio((0, 4, 0)) == 0.0


@pytest.mark.parametrize("H,W,d", [(256, 256, 7), (512, 512, 14), (512, 1024, 23), (1024, 2048, 46), (10, 10, 1),
                                   (1, 1, 1), (30, 40, 1), (40, 40, 1), (1, 100, 2)])
def test_dilation_rule(H, W, d):
    import dct_b200
    assert OB.dilation_for(H, W) == d
    assert dct_b200.metrics.boundary_dilation(H, W) == d


def test_dilation_rounds_half_to_even():
    import dct_b200
    f = dct_b200.metrics.boundary_dilation
    # ratio * 5 (a 3 x 4 image) lands on x.5 exactly: Python's round goes to the even neighbour
    assert f(3, 4, 0.5) == 2 == round(2.5) and f(3, 4, 0.7) == 4 == round(3.5)
    assert f(3, 4, 0.01) == 1   # the minimum of 1


def test_argument_parsing():
    import dct_b200
    f = dct_b200.metrics.boundary_dilation
    assert f(512, 1024, dilation=5) == 5 and f(512, 1024, 0.05) == 57
    for bad in (0.0, -0.1, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            f(64, 64, bad)
    for bad in (0, -2, 1.5):
        with pytest.raises(ValueError):
            f(64, 64, dilation=bad)
    ign = dct_b200.metrics._ignore_arg
    assert ign(None, 19) == -1 and ign(255, 19) == 255 and ign(19, 19) == 19
    for bad in (0, 18, -1, 2.5):
        with pytest.raises(ValueError):
            ign(bad, 19)
    with pytest.raises(ValueError):
        dct_b200.BoundaryIoUMeter(4, dilation=0)
    with pytest.raises(ValueError):
        dct_b200.BoundaryIoUMeter(4, ignore_index=2)
    for bad in (0, 65, 2.5):
        with pytest.raises(ValueError):
            dct_b200.BoundaryIoUMeter(bad)
    assert dct_b200.BoundaryIoUMeter(64).C == 64


def test_boundary_iou_scratch_bytes_and_limits():
    import dct_b200
    h = dct_b200._lib.lib()

    def a256(v):
        return (v + 255) // 256 * 256

    for C, B, H, W in [(4, 10, 256, 256), (19, 3, 17, 23), (2, 1, 1, 1), (19, 4, 1024, 2048), (64, 1, 1, 2 ** 31 - 1)]:
        assert h.dct_boundary_iou_scratch_bytes(C, B, H, W) == a256(2 * B * H * W) + a256(24 * B * C)
    assert h.dct_boundary_iou_scratch_bytes(65, 1, 8, 8) == 0
    assert h.dct_boundary_iou_scratch_bytes(0, 1, 8, 8) == 0
    for shape in [(1, 1, 2 ** 31), (2 ** 31, 1, 1), (1, 2 ** 31, 1), (2, 2 ** 15, 2 ** 15), (0, 8, 8), (1, 0, 8),
                  (1, 8, 0), (1, 2 ** 32, 2 ** 32)]:
        assert h.dct_boundary_iou_scratch_bytes(4, *shape) == 0, shape
    for shape in [(2 ** 31 - 1, 1, 1), (1, 2 ** 31 - 1, 1), (1, 46340, 46340), (2, 2 ** 15, 2 ** 15 - 1)]:
        assert h.dct_boundary_iou_scratch_bytes(4, *shape) > 0, shape


def test_boundary_iou_abi_rejects_bad_arguments():
    """Argument checks run on the host before anything is launched (no GPU needed); codes as dct_surface_dice_i64."""
    import dct_b200
    h = dct_b200._lib.lib()
    fake = 1 << 20   # aligned non-null stand-ins: rejected before any dereference
    f = h.dct_boundary_iou_i64
    assert f(None, fake, 4, 2, 8, 8, 2, -1, fake, None, None, fake, None) == -1
    assert f(fake, None, 4, 2, 8, 8, 2, -1, fake, None, None, fake, None) == -1
    assert f(fake, fake, 4, 2, 8, 8, 2, -1, None, fake, None, fake, None) == -1
    assert f(fake, fake, 4, 2, 8, 8, 2, -1, fake, fake, fake, None, None) == -1
    for C, B, H, W in [(0, 2, 8, 8), (4, 0, 8, 8), (4, 2, 0, 8), (4, 2, 8, -1)]:
        assert f(fake, fake, C, B, H, W, 2, -1, fake, None, None, fake, None) == -1
    for d in (0, -1, -(2 ** 40)):
        assert f(fake, fake, 4, 2, 8, 8, d, -1, fake, None, None, fake, None) == -1
    for ignore in (0, 3):
        assert f(fake, fake, 4, 2, 8, 8, 2, ignore, fake, None, None, fake, None) == -1
    assert f(fake, fake, 65, 2, 8, 8, 2, 255, fake, None, None, fake, None) == -2
    assert f(fake, fake, 4, 1, 2 ** 16, 2 ** 15, 2, 255, fake, None, None, fake, None) == -2
    assert f(fake + 4, fake, 4, 2, 8, 8, 2, -1, fake, None, None, fake, None) == -3
    assert f(fake, fake + 4, 4, 2, 8, 8, 2, -1, fake, None, None, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 2, -1, fake + 2, None, None, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 2, -1, fake, fake + 4, None, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 2, -1, fake, None, fake + 2, fake, None) == -3
    assert f(fake, fake, 4, 2, 8, 8, 2, -1, fake, None, None, fake + 128, None) == -3
