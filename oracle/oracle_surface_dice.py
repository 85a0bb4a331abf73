"""Normalized surface Dice oracle (test infrastructure): surface Dice at a tolerance restated from the distances of
``oracle_surface.surface_distances`` (scipy's EDT), and a brute-force form it is checked against.

Border-pixel form: every border pixel counts once (MONAI's ``compute_surface_dice`` with ``use_subvoxels=False`` works
this way; this restatement is written from the definition below and not checked against MONAI).  Borders, grids and
spacing are those of ``oracle_hausdorff``.  With ``S_pg`` the distances from each border pixel of ``a`` (prediction) to
``border(g)`` (label) and ``S_gp`` the other way, a distance to an empty border being +inf:
  ``W_pg = #{s in S_pg : s <= tol}``, ``W_gp`` likewise;
  ``nsd = (W_pg + W_gp) / (|S_pg| + |S_gp|)``: NaN only when both borders are empty, 0 when exactly one is;
  ``overlap_pg = W_pg / |S_pg|``, ``overlap_gp = W_gp / |S_gp|``: each NaN when its denominator is 0.
"""
import numpy as np
from scipy.spatial.distance import cdist

from oracle_hausdorff import border
from oracle_surface import surface_distances

KEYS = ("nsd", "overlap_pg", "overlap_gp")


def _to_border(a: np.ndarray, g: np.ndarray, spacing) -> np.ndarray:
    """Distances from each border pixel of ``a`` to ``border(g)``; +inf when ``g`` is empty."""
    if not g.any():
        return np.full(int(border(a).sum()), np.inf)
    return surface_distances(a, g, spacing)


def _to_border_brute(a: np.ndarray, g: np.ndarray, spacing) -> np.ndarray:
    sp = np.ones(a.ndim) if spacing is None else np.asarray(spacing, dtype=np.float64)
    pa, pg = np.argwhere(border(a)) * sp, np.argwhere(border(g)) * sp
    if len(pg) == 0:
        return np.full(len(pa), np.inf)
    return cdist(pa, pg).min(1) if len(pa) else np.zeros(0)


def _counts(s_pg: np.ndarray, s_gp: np.ndarray, tol: float):
    return int(np.count_nonzero(s_pg <= tol)), s_pg.size, int(np.count_nonzero(s_gp <= tol)), s_gp.size


def ratios(counts):
    """(nsd, overlap_pg, overlap_gp) in double from the counts ``(W_pg, |S_pg|, W_gp, |S_gp|)``."""
    w_pg, n_pg, w_gp, n_gp = (int(v) for v in counts)
    nan = float("nan")
    return ((w_pg + w_gp) / (n_pg + n_gp) if n_pg + n_gp else nan, w_pg / n_pg if n_pg else nan,
            w_gp / n_gp if n_gp else nan)


def surface_dice_binary(a: np.ndarray, g: np.ndarray, tol: float, spacing=None):
    """Counts ``(W_pg, |S_pg|, W_gp, |S_gp|)`` of prediction ``a`` against label ``g`` at tolerance ``tol``."""
    a, g = a.astype(bool), g.astype(bool)
    return _counts(_to_border(a, g, spacing), _to_border(g, a, spacing), tol)


def surface_dice_binary_brute(a: np.ndarray, g: np.ndarray, tol: float, spacing=None):
    """The same from the border coordinates: all pairwise distances (argwhere + cdist)."""
    a, g = a.astype(bool), g.astype(bool)
    return _counts(_to_border_brute(a, g, spacing), _to_border_brute(g, a, spacing), tol)


def surface_dice(pred: np.ndarray, gt: np.ndarray, C: int, tol, method: str = "2d", spacing=None,
                 brute: bool = False) -> dict:
    """``{'nsd', 'overlap_pg', 'overlap_gp'}``, each float64 ``[rows, C]``, and ``'counts'`` int64 ``[rows, C, 4]`` =
    ``(W_pg, |S_pg|, W_gp, |S_gp|)`` for integer maps ``[B,H,W]`` (rows = B for '2d', 1 for '3d'); ``tol`` is a scalar or
    one value per class."""
    assert method in ("2d", "3d") and pred.shape == gt.shape and pred.ndim == 3
    tols = np.broadcast_to(np.asarray(tol, dtype=np.float64), (C,))
    f = surface_dice_binary_brute if brute else surface_dice_binary
    grids = [(pred, gt)] if method == "3d" else [(pred[b], gt[b]) for b in range(pred.shape[0])]
    counts = np.array([[f(p == c, g == c, float(tols[c]), spacing) for c in range(C)] for p, g in grids],
                      dtype=np.int64).reshape(len(grids), C, 4)
    r = np.array([[ratios(counts[i, c]) for c in range(C)] for i in range(len(grids))],
                 dtype=np.float64).reshape(len(grids), C, 3)
    out = {k: r[:, :, i] for i, k in enumerate(KEYS)}
    out["counts"] = counts
    return out


def distances(pred: np.ndarray, gt: np.ndarray, C: int, method: str = "2d", spacing=None):
    """Every distance the counts compare, per (row, class): ``[[(S_pg, S_gp) for c] for row]`` (float64 arrays)."""
    grids = [(pred, gt)] if method == "3d" else [(pred[b], gt[b]) for b in range(pred.shape[0])]
    return [[(_to_border(p == c, g == c, spacing), _to_border(g == c, p == c, spacing)) for c in range(C)]
            for p, g in grids]
