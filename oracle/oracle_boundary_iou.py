"""Boundary IoU oracle (test infrastructure): the definition's own code, a scipy restatement and a brute-force window
check, and the per-(image, class) counts and ratios of ``dct_boundary_iou_i64``.

Definition (Cheng et al., CVPR 2021; ``mask_to_boundary`` of the authors' boundary-iou-api): the band of width ``d`` of a
binary mask ``M`` is ``M - erode(pad(M, 1, 0), ones((3, 3)), iterations=d)[1:H+1, 1:W+1]``: the pixels of ``M`` whose
(2d+1) x (2d+1) square is not entirely on the grid and inside ``M``.  ``scipy.ndimage.minimum_filter(M, size=2d+1,
mode='constant', cval=0)`` is the same erosion in one step.
"""
import math

import numpy as np
from scipy.ndimage import minimum_filter


def dilation_for(H: int, W: int, ratio: float = 0.02) -> int:
    """``mask_to_boundary``'s band width for an ``H x W`` image: ``max(1, int(round(ratio * sqrt(H**2 + W**2))))``."""
    return max(1, int(round(ratio * np.sqrt(H ** 2 + W ** 2))))


def mask_to_boundary_cv2(mask: np.ndarray, d: int) -> np.ndarray:
    """The definition's code (boundary-iou-api ``mask_to_boundary`` with ``dilation = d``), on a uint8 mask."""
    import cv2
    h, w = mask.shape
    m = mask.astype(np.uint8)
    new_mask = cv2.copyMakeBorder(m, 1, 1, 1, 1, cv2.BORDER_CONSTANT, value=0)
    kernel = np.ones((3, 3), dtype=np.uint8)
    new_mask_erode = cv2.erode(new_mask, kernel, iterations=d)
    return (m - new_mask_erode[1: h + 1, 1: w + 1]).astype(bool)


def mask_to_boundary(mask: np.ndarray, d: int) -> np.ndarray:
    """The same band with scipy: ``M & ~minimum_filter(M, 2d+1, constant 0)``."""
    m = mask.astype(np.uint8)
    return m.astype(bool) & ~minimum_filter(m, size=2 * d + 1, mode="constant", cval=0).astype(bool)


def mask_to_boundary_brute(mask: np.ndarray, d: int) -> np.ndarray:
    """The same band by the window test at every pixel of the mask."""
    m = mask.astype(bool)
    h, w = m.shape
    out = np.zeros_like(m)
    for y, x in np.argwhere(m):
        inside = y - d >= 0 and y + d < h and x - d >= 0 and x + d < w and m[y - d: y + d + 1, x - d: x + d + 1].all()
        out[y, x] = not inside
    return out


def ratio(counts) -> float:
    """``I / (G + P - I)`` in double from ``(I, G, P)``; NaN for an empty union."""
    i, g, p = (int(v) for v in counts)
    u = g + p - i
    return i / u if u else math.nan


def boundary_iou(pred: np.ndarray, gt: np.ndarray, C: int, d: int, ignore_index=None, band=mask_to_boundary) -> dict:
    """``{'counts': int64 [B, C, 3] = (I, G, P), 'biou': float64 [B, C]}`` for integer maps ``[B, H, W]``: per image and
    class, ``I = |band(P) & band(G) & valid|``, ``G = |band(G)|``, ``P = |band(P) & valid|`` with ``valid = gt !=
    ignore_index``; values outside ``[0, C)`` belong to no class."""
    assert pred.shape == gt.shape and pred.ndim == 3
    B = pred.shape[0]
    counts = np.zeros((B, C, 3), np.int64)
    for b in range(B):
        valid = np.ones(gt[b].shape, bool) if ignore_index is None else gt[b] != ignore_index
        for c in range(C):
            bp, bg = band(pred[b] == c, d), band(gt[b] == c, d)
            counts[b, c] = (np.count_nonzero(bp & bg & valid), np.count_nonzero(bg), np.count_nonzero(bp & valid))
    biou = np.array([[ratio(counts[b, c]) for c in range(C)] for b in range(B)], np.float64).reshape(B, C)
    return {"counts": counts, "biou": biou}
