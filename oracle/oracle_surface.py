"""Surface-distance oracle (test infrastructure): ``medpy.metric.binary`` ``hd95``, ``asd`` and ``assd`` restated with scipy,
a brute-force form they are checked against, and numpy's 95th percentile written out as scalar arithmetic.

medpy (``medpy/metric/binary.py``, connectivity 1), with ``__surface_distances(result, reference)`` the distances from each
border pixel of ``result`` to the border of ``reference`` (borders and spacing as in ``oracle_hausdorff``):
  ``hd95(result, reference)`` = ``np.percentile(np.hstack((sds(result, reference), sds(reference, result))), 95)``;
  ``asd(result, reference)``  = ``sds(result, reference).mean()`` (directional);
  ``assd(result, reference)`` = ``np.mean((asd(result, reference), asd(reference, result)))``.
medpy raises ``RuntimeError`` when either mask is empty; here every value is NaN then.  Per class of integer maps, rows and
classes are those of ``oracle_hausdorff.hausdorff``.
"""
import math

import numpy as np
from scipy.ndimage import distance_transform_edt
from scipy.spatial.distance import cdist

from oracle_hausdorff import border

KEYS = ("hd", "hd95", "asd", "assd")


def surface_distances(a: np.ndarray, g: np.ndarray, spacing=None) -> np.ndarray:
    """medpy's ``__surface_distances(a, g, spacing, 1)``: float64 distances from each border pixel of ``a`` to ``border(g)``."""
    sp = None if spacing is None else np.asarray(spacing, dtype=np.float64)
    return distance_transform_edt(~border(g), sampling=sp)[border(a)]


def percentile95(x) -> float:
    """``np.percentile(x, 95)`` (method 'linear') as scalar double arithmetic: the virtual index is ``(n - 1) * 0.95``."""
    s = np.sort(np.asarray(x, dtype=np.float64).ravel())
    n = s.size
    v = (n - 1) * 0.95
    lo = math.floor(v)
    t = v - lo
    hi = min(lo + 1, n - 1)
    a, b = float(s[lo]), float(s[hi])
    d = b - a
    return b - d * (1 - t) if t >= 0.5 else a + d * t


def _metrics(s_pg: np.ndarray, s_gp: np.ndarray):
    return (float(max(s_pg.max(), s_gp.max())), float(np.percentile(np.hstack((s_pg, s_gp)), 95)),
            float(s_pg.mean()), float(np.mean((s_pg.mean(), s_gp.mean()))))


def surface_binary(a: np.ndarray, g: np.ndarray, spacing=None):
    """(hd, hd95, asd, assd) of medpy for result ``a`` and reference ``g``; NaN for an empty mask."""
    a, g = a.astype(bool), g.astype(bool)
    if not a.any() or not g.any():
        return (float("nan"),) * 4
    return _metrics(surface_distances(a, g, spacing), surface_distances(g, a, spacing))


def surface_binary_brute(a: np.ndarray, g: np.ndarray, spacing=None):
    """The same from the border coordinates: all pairwise distances (argwhere + cdist)."""
    a, g = a.astype(bool), g.astype(bool)
    if not a.any() or not g.any():
        return (float("nan"),) * 4
    sp = np.ones(a.ndim) if spacing is None else np.asarray(spacing, dtype=np.float64)
    d = cdist(np.argwhere(border(a)) * sp, np.argwhere(border(g)) * sp)
    return _metrics(d.min(1), d.min(0))


def surface(pred: np.ndarray, gt: np.ndarray, C: int, method: str = "2d", spacing=None, brute: bool = False) -> dict:
    """``{'hd', 'hd95', 'asd', 'assd'}``, each float64 ``[rows, C]`` for integer maps ``[B,H,W]`` (rows = B for '2d', 1 for
    '3d')."""
    assert method in ("2d", "3d") and pred.shape == gt.shape and pred.ndim == 3
    f = surface_binary_brute if brute else surface_binary
    grids = [(pred, gt)] if method == "3d" else [(pred[b], gt[b]) for b in range(pred.shape[0])]
    v = np.array([[f(p == c, g == c, spacing) for c in range(C)] for p, g in grids], dtype=np.float64)
    return {k: v[:, :, i] for i, k in enumerate(KEYS)}
